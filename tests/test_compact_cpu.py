"""Compaction (turdb_cuda_index_compact) without a device: hand-worked known answers for the CPU reference's restatement
of the rule (tests/compact_reference.py), its recall against the filtered traversal it replaces, and the C entry's and
the wrapper's behaviour before any device work."""
import ctypes as C

import numpy as np
import pytest

import compact_reference
from oracle import binding as ob
from turdb_b200 import _lib
from turdb_b200 import datasets as ds
from turdb_b200.hnsw import CudaHnswIndex, DistanceFunction, visibility_bitmap

INV = ob.INVALID


def graph(points, levels, l0, upper=None, entry=0, max_level=0):
    """Graph arrays from 2-d integer points (squared distances are exact), level-0 lists and {node: [list per level]}."""
    n = len(points)
    levels = np.array(levels, np.uint8)
    up_base = np.full(n, INV, np.uint32)
    slots = []
    for i in range(n):
        if levels[i]:
            up_base[i] = len(slots)
            slots += [(upper or {}).get(i, [[]] * levels[i])[l] for l in range(levels[i])]
    l0_adj = np.full((n, 32), INV, np.uint32)
    for i, lst in enumerate(l0):
        l0_adj[i, :len(lst)] = lst
    up_adj = np.full((len(slots), 16), INV, np.uint32)
    for s, lst in enumerate(slots):
        up_adj[s, :len(lst)] = lst
    return dict(vectors=np.array(points, np.float32), row_ids=np.arange(n, dtype=np.uint64) + 100, levels=levels,
                l0_adj=l0_adj, l0_cnt=np.array([len(x) for x in l0], np.uint8), up_base=up_base, up_adj=up_adj,
                up_cnt=np.array([len(x) for x in slots], np.uint8), entry=entry, max_level=max_level)


def lists(arrays, level0=True):
    adj, cnt = (arrays["l0_adj"], arrays["l0_cnt"]) if level0 else (arrays["up_adj"], arrays["up_cnt"])
    return [adj[i, :cnt[i]].tolist() for i in range(len(cnt))]


def compact(arrays, dead):
    return compact_reference.compact(arrays, ~np.isin(np.arange(len(arrays["levels"])), dead))


def test_deleted_neighbour_refills_the_list():
    # 0 (0,0) lists [4, 1]; the deleted 1 lists [2, 0, 3].  C for 0 = [4 (9), 2 (4), 3 (9)] -> sorted 2, 4, 3 (the tie
    # keeps C's order); the walk keeps 2, drops 4 (|4-2|^2 = 1 < 9), keeps 3 (13 >= 9); the back-fill appends 4.
    g = graph([(0, 0), (5, 5), (2, 0), (0, 3), (3, 0), (10, 10)], [0] * 6,
              [[4, 1], [2, 0, 3], [1], [1, 0], [0, 5], [4]])
    a, o2n = compact(g, [1])
    assert o2n.tolist() == [0, INV, 1, 2, 3, 4]
    # old lists: 0 -> [2, 3, 4]; 2 -> C [0 (4), 3 (13)] walk keeps 0, drops 3 (9 < 13), back-fill 3; 3 -> C [0 (9), 2 (13)]
    # keeps 0, drops 2 (4 < 13), back-fill 2; 4 and 5 hold no deleted id: verbatim
    assert lists(a) == [[1, 2, 3], [0, 2], [0, 1], [0, 4], [3]]
    assert a["row_ids"].tolist() == [100, 102, 103, 104, 105]
    assert a["vectors"][1].tolist() == [2, 0]
    assert (a["entry"], a["max_level"], a["up_cnt"].size) == (0, 0, 0)


def test_deleted_entry_one_way_link_and_upper_lists():
    # levels 2 1 0 1 0; the entry 0 and node 2 are deleted.  Node 1's level-1 list holds 2, which lacks level 1 (the
    # insert path's one-way link): 2 contributes nothing there.
    g = graph([(0, 0), (1, 0), (2, 0), (0, 1), (5, 5)], [2, 1, 0, 1, 0],
              [[1, 2, 3], [0, 2], [1, 0, 4], [0, 4], [2, 3]],
              upper={0: [[1, 3], []], 1: [[2, 0, 3]], 3: [[1]]}, entry=0, max_level=2)
    a, o2n = compact(g, [0, 2])
    assert o2n.tolist() == [INV, 0, INV, 1, 2]
    # level 0: 1 -> C [3 (2), 4 (41)], 4 kept (|4-3|^2 = 41 is not < 41); 3 -> C [4 (41), 1 (2)] -> [1, 4];
    # 4 -> C [3 (41), 1 (41)] (tie: C's order), 1 dropped (2 < 41) and back-filled
    assert lists(a) == [[1, 2], [0, 2], [1, 0]]
    # level 1: 1 -> C [3] (2 lacks the level, 0's level-1 list adds only 1 itself and 3 again); 3 -> [1] verbatim
    assert lists(a, level0=False) == [[1], [0]]
    assert a["up_base"].tolist() == [0, 1, INV] and a["levels"].tolist() == [1, 1, 0]
    # the deleted entry: the live nodes of the highest level are old 1 and 3, the lowest new id wins
    assert (a["entry"], a["max_level"]) == (0, 1)


def test_every_node_deleted_gives_an_empty_graph():
    g = graph([(0, 0), (1, 0), (2, 0)], [1, 0, 0], [[1, 2], [0], [0]], upper={0: [[]]}, entry=0, max_level=1)
    a, o2n = compact(g, [0, 1, 2])
    assert o2n.tolist() == [INV] * 3
    assert (len(a["levels"]), a["entry"], a["max_level"]) == (0, INV, 0)
    assert a["up_cnt"].size == 0 and a["l0_adj"].shape == (0, 32)
    empty = ob.OracleGraph.from_arrays(a)  # what the device's empty index is checked against
    assert (empty.n, empty.entry, empty.max_level) == (0, INV, 0)


def test_nothing_deleted_changes_nothing(small_graph):
    _, arrays = small_graph
    a, o2n = compact(arrays, [])
    assert np.array_equal(o2n, np.arange(len(o2n), dtype=np.uint32))
    for key in ("vectors", "row_ids", "levels", "l0_adj", "l0_cnt", "up_base", "up_adj", "up_cnt", "entry", "max_level"):
        assert np.array_equal(a[key], arrays[key]), key


def test_compacted_graph_keeps_the_filtered_recall(small_graph):
    # measured on this corpus (1000 queries): filtered 0.9986, compacted 0.9985 at 10 % deleted
    g, arrays = small_graph
    x = arrays["vectors"]
    dead = np.random.default_rng(3).random(g.n) < 0.1
    live = np.flatnonzero(~dead)
    q = ds.gaussian_latent(300, 128, seed=81)
    d2 = ((q[:, None, :] - x[None, live, :]) ** 2).sum(-1)
    truth = live[np.argsort(d2, axis=1)[:, :10]]
    words = visibility_bitmap(~dead)
    _, filtered, _, _, _ = g.search(q, 10, 64, ob.L2, visible=words, n_threads=8)
    a, o2n = compact(arrays, np.flatnonzero(dead))
    c = ob.OracleGraph.from_arrays(a)
    assert np.array_equal(o2n[live], np.arange(len(live))) and (o2n[dead] == INV).all()
    _, compacted, _, _, _ = c.search(q, 10, 64, ob.L2, n_threads=8)
    compacted = np.where(compacted != INV, live[np.minimum(compacted, len(live) - 1)], -1)

    def recall(got):
        return np.mean([len(set(got[i].tolist()) & set(truth[i].tolist())) / 10 for i in range(len(q))])
    assert recall(compacted) >= recall(filtered) - 0.01
    # every list refers to live nodes only, and no list refers to its owner
    for i, lst in enumerate(lists(a)):
        assert i not in lst and all(v < len(live) for v in lst)


def test_compact_null_index_is_an_invalid_argument():
    L = _lib.load()
    out = np.full(2, 7, np.uint32)
    n = C.c_uint64(9)
    assert L.turdb_cuda_index_compact(None, out.ctypes.data_as(C.POINTER(C.c_uint32)), C.byref(n)) == \
        _lib.ERR_INVALID_ARGUMENT
    assert b"idx is null" in L.turdb_cuda_last_error()
    assert out.tolist() == [7, 7] and n.value == 9  # nothing written on failure
    assert L.turdb_cuda_index_compact(None, None, None) == _lib.ERR_INVALID_ARGUMENT


def test_wrapper_returns_the_map_and_updates_the_node_count(monkeypatch):
    seen = {}

    class Fake:
        def turdb_cuda_index_compact(self, h, ptr, out_n):
            seen["called"] = True
            np.ctypeslib.as_array(ptr, shape=(5,))[:] = [0, INV, 1, INV, 2]
            out_n._obj.value = 3
            return _lib.OK

    monkeypatch.setattr(_lib, "load", lambda: Fake())
    idx = CudaHnswIndex(None, 8, 5, DistanceFunction.L2, 0)
    o2n = idx.compact()
    assert seen["called"] and o2n.dtype == np.uint32 and o2n.tolist() == [0, INV, 1, INV, 2]
    assert idx.n == 3
