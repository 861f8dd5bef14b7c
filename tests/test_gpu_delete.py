"""Deleting rows from a resident index (turdb_cuda_index_delete): a deleted row is a row the table no longer holds.
Traversals must equal search_filtered with visibility `live` (a twin index without deletions searched with that bitmap,
and the oracle); every exact and SQL statement must equal the same call on an index holding only the live rows, row for
row and bit for bit; insert must ignore deletions; an index without deletions must answer exactly as before."""
import ctypes as C
import re

import numpy as np
import pytest
import torch

from oracle import binding as ob
from turdb_b200 import _lib
from turdb_b200 import datasets as ds
from turdb_b200.hnsw import INVALID_ROW, CudaHnswIndex, DistanceFunction, shards_search_batch, visibility_bitmap
from turdb_b200.sql_operator import (RangeCmp, VectorOp, VectorRangeScanBatch, VectorRangeTopKBatch, VectorScanBatch,
                                     VectorTopKExec)

pytestmark = pytest.mark.gpu

GRAPH_KEYS = ("vectors", "row_ids", "levels", "l0_adj", "l0_cnt", "up_base", "up_adj", "up_cnt")
NEAR = [(VectorOp.L2Distance, RangeCmp.Lt), (VectorOp.L2Distance, RangeCmp.Le), (VectorOp.CosineDistance, RangeCmp.Lt),
        (VectorOp.CosineDistance, RangeCmp.Le), (VectorOp.InnerProduct, RangeCmp.Gt), (VectorOp.InnerProduct, RangeCmp.Ge)]


def table_index(x, row_ids=None):
    """A table without an HNSW graph: the exact scan only needs the arena (entry = none)."""
    n = x.shape[0]
    g = dict(vectors=x, row_ids=np.arange(n, dtype=np.uint64) if row_ids is None else row_ids,
             levels=np.zeros(n, np.uint8), l0_adj=np.full((n, 32), 0xFFFFFFFF, np.uint32), l0_cnt=np.zeros(n, np.uint8),
             up_base=np.full(n, 0xFFFFFFFF, np.uint32), up_adj=np.zeros((0, 16), np.uint32), up_cnt=np.zeros(0, np.uint8),
             entry=0 if n else 0xFFFFFFFF, max_level=0)
    return CudaHnswIndex.from_graph(g)


def deleted_mask(n, frac, seed):
    """bool[n]: True = deleted.  frac 1.0 deletes every row."""
    return np.random.default_rng(seed).random(n) < frac if frac < 1.0 else np.ones(n, bool)


def same_bits(a, b, what=""):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    assert a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8)), what


def same_traversal(got, want):
    """search_batch outputs: rows, nodes, distance bits, counts and the n_dist / n_expanded statistics."""
    for i, what in enumerate(("rows", "nodes", "dist", "counts")):
        same_bits(got[i], want[i], what)
    for f in ("n_dist", "n_expanded"):
        assert np.array_equal(got[4][f], want[4][f]), f


def same_as_oracle(got, cpu):
    assert np.array_equal(got[3], cpu[3]), "counts differ"
    for i in range(len(got[3])):
        c = cpu[3][i]
        assert np.array_equal(got[1][i][:c], cpu[1][i][:c]), i
        assert np.array_equal(got[2][i][:c].view(np.uint32), cpu[2][i][:c].view(np.uint32)), i
    for f in ("n_dist", "n_expanded"):
        assert np.array_equal(got[4][f], cpu[4][f]), f


def fallbacks(capfd, what):
    """Statements the streaming scan redid in the last call, from its TURDB_EXACT_VERBOSE line."""
    m = re.findall(rf"\[turdb {what}\] statements=(\d+) fallback=(\d+)", capfd.readouterr().err)
    assert m, "no TURDB_EXACT_VERBOSE line"
    return int(m[-1][1])


# ---- 1. the reference's own answer -----------------------------------------------------------------------------------
def test_knn_search_after_delete_excludes_deleted(gpu_required):
    # knn_search_after_delete_excludes_deleted, tests/hnsw_integration.rs:238-256: DELETE the row with id 1
    ids = np.array([1, 2, 3], np.uint64)
    x = np.array([[0.1] * 4, [0.5] * 4, [0.9] * 4], np.float32)
    idx = table_index(x, ids)
    assert idx.delete([0]) == 1
    ex = VectorTopKExec(idx, VectorOp.L2Distance, "[0.1, 0.1, 0.1, 0.1]", limit=2)
    ex.open()
    assert [ex.next()[0], ex.next()[0]] == [2, 3] and ex.next() is None
    idx.close()


# ---- 2. traversal = search_filtered over `live` ----------------------------------------------------------------------
@pytest.mark.parametrize("frac", [0.0, 0.01, 0.5, 1.0])
@pytest.mark.parametrize("metric", [ob.L2, ob.COSINE, ob.IP])
def test_traversal_is_search_filtered_over_live(gpu_required, small_graph, frac, metric):
    g, arrays = small_graph
    dead = deleted_mask(g.n, frac, int(frac * 1000) + metric)
    q = ds.gaussian_latent(96, 128, seed=51)
    idx, twin = CudaHnswIndex.from_graph(arrays), CudaHnswIndex.from_graph(arrays)
    assert idx.delete(np.flatnonzero(dead)) == int(dead.sum())
    words = visibility_bitmap(~dead) if dead.any() else None  # nothing deleted: the unfiltered search
    cpu = g.search(q, 10, 64, metric, visible=words, n_threads=8)
    for form in (1, 2):
        idx.set_traversal_form(form)
        twin.set_traversal_form(form)
        got = idx.search_batch(q, 10, 64, DistanceFunction(metric))
        same_traversal(got, twin.search_batch(q, 10, 64, DistanceFunction(metric), visible=words))
        same_as_oracle(got, cpu)
        assert not dead[got[1][got[1] != 0xFFFFFFFF]].any()
    if frac == 1.0:
        assert (got[3] == 0).all()
    idx.close()
    twin.close()


def test_deleted_entry_node_and_caller_bitmap(gpu_required, small_graph):
    g, arrays = small_graph
    dead = deleted_mask(g.n, 0.1, 5)
    dead[arrays["entry"]] = True
    vis = np.random.default_rng(6).random(g.n) < 0.6
    q = ds.gaussian_latent(96, 128, seed=52)
    idx, twin = CudaHnswIndex.from_graph(arrays), CudaHnswIndex.from_graph(arrays)
    idx.delete(np.flatnonzero(dead))
    for form in (1, 2):
        idx.set_traversal_form(form)
        twin.set_traversal_form(form)
        for caller, words in ((None, visibility_bitmap(~dead)), (visibility_bitmap(vis), visibility_bitmap(vis & ~dead))):
            got = idx.search_batch(q, 10, 48, visible=caller)
            same_traversal(got, twin.search_batch(q, 10, 48, visible=words))
            same_as_oracle(got, g.search(q, 10, 48, ob.L2, visible=words, n_threads=8))
    idx.close()
    twin.close()


def test_device_and_sq8_traversals(gpu_required, small_graph):
    g, arrays = small_graph
    dead = deleted_mask(g.n, 0.2, 7)
    q = ds.gaussian_latent(64, 128, seed=53)
    idx, twin = CudaHnswIndex.from_graph(arrays), CudaHnswIndex.from_graph(arrays)
    idx.delete(np.flatnonzero(dead))
    idx.enable_sq8()
    twin.enable_sq8()
    dq = torch.from_numpy(q).cuda()
    d_vis = torch.from_numpy(visibility_bitmap(~dead).view(np.int64)).cuda()
    d_caller = torch.from_numpy(visibility_bitmap(np.arange(g.n) % 3 != 0).view(np.int64)).cuda()
    d_both = torch.from_numpy(visibility_bitmap((np.arange(g.n) % 3 != 0) & ~dead).view(np.int64)).cuda()
    stream = torch.cuda.current_stream().cuda_stream

    def run(ix, fn, visible):
        out = [torch.zeros((64, 10), dtype=torch.int64, device="cuda"), torch.zeros((64, 10), dtype=torch.float32, device="cuda"),
               torch.zeros(64, dtype=torch.int32, device="cuda"), torch.zeros((64, 10), dtype=torch.int32, device="cuda"),
               torch.zeros((64, 4), dtype=torch.int32, device="cuda")]
        getattr(ix, fn)(dq.data_ptr(), 64, 10, 64, 0, out[0].data_ptr(), out[1].data_ptr(), out[2].data_ptr(),
                        d_nodes=out[3].data_ptr(), d_stats=out[4].data_ptr(), stream=stream,
                        d_visible=0 if visible is None else visible.data_ptr())
        torch.cuda.synchronize()
        return [t.cpu().numpy() for t in out]

    for fn in ("search_batch_device", "search_batch_sq8_device"):
        for mine, theirs in ((None, d_vis), (d_caller, d_both)):
            for a, b in zip(run(idx, fn, mine), run(twin, fn, theirs)):
                same_bits(a, b, fn)
    idx.close()
    twin.close()


def test_shards_search_batch(gpu_required, small_graph):
    g, arrays = small_graph
    half = g.n // 2
    parts = []
    for lo, hi in ((0, half), (half, g.n)):
        x = arrays["vectors"][lo:hi]
        parts.append((CudaHnswIndex.build(x, arrays["row_ids"][lo:hi], max_batch=256),
                      CudaHnswIndex.build(x, arrays["row_ids"][lo:hi], max_batch=256), deleted_mask(hi - lo, 0.3, lo + 1)))
    q = ds.gaussian_latent(64, 128, seed=54)
    for idx, _, dead in parts:
        idx.delete(np.flatnonzero(dead))
    rows, dist, counts = shards_search_batch([p[0] for p in parts], q, 10, 64)
    lists = [twin.search_batch(q, 10, 64, visible=visibility_bitmap(~dead)) for _, twin, dead in parts]
    for i in range(len(q)):
        pairs = sorted((float(l[2][i, j]), int(l[0][i, j])) for l in lists for j in range(int(l[3][i])))[:10]
        assert counts[i] == len(pairs)
        assert [r for _, r in pairs] == rows[i, :counts[i]].tolist()
        assert np.array_equal(np.array([d for d, _ in pairs], np.float32).view(np.uint32), dist[i, :counts[i]].view(np.uint32))
    for idx, twin, _ in parts:
        idx.close()
        twin.close()


# ---- 3. without deletions nothing changes ------------------------------------------------------------------------------
def test_empty_delete_changes_nothing(gpu_required, small_graph):
    g, arrays = small_graph
    q = ds.gaussian_latent(64, 128, seed=55)
    idx = CudaHnswIndex.from_graph(arrays)
    before = (idx.search_batch(q, 10, 64), idx.bruteforce_topk(q, 10),
              VectorScanBatch(idx, VectorOp.L2Distance, 10).execute(q),
              VectorRangeScanBatch(idx, VectorOp.L2Distance, RangeCmp.Lt, 10).execute(q, np.full(64, 9.0)))
    nbytes = idx.info()["device_bytes"]
    assert idx.delete([]) == 0 and idx.delete(np.zeros(0, np.uint32)) == 0
    after = (idx.search_batch(q, 10, 64), idx.bruteforce_topk(q, 10),
             VectorScanBatch(idx, VectorOp.L2Distance, 10).execute(q),
             VectorRangeScanBatch(idx, VectorOp.L2Distance, RangeCmp.Lt, 10).execute(q, np.full(64, 9.0)))
    for b, a in zip(before, after):
        for x, y in zip(b, a):
            same_bits(x, y)
    assert idx.info()["device_bytes"] == nbytes
    idx.close()


# ---- 4. exact and SQL statements = the same call on the live rows ----------------------------------------------------
def approx_values(x, q, op):
    """float64 values for choosing radii (not the parity values)."""
    x64, q64 = x.astype(np.float64), q.astype(np.float64)
    dot = q64 @ x64.T
    if op == VectorOp.InnerProduct:
        return dot
    xn, qn = (x64 ** 2).sum(axis=1), (q64 ** 2).sum(axis=1)
    if op == VectorOp.L2Distance:
        return np.sqrt(np.maximum(qn[:, None] + xn[None, :] - 2 * dot, 0))
    return 1 - dot / np.maximum(np.sqrt(np.outer(qn, xn)), 1e-30)


def compare_statements(idx, twin, x, rid, dead, q, grid=((10, 0), (5, 7), (1, 0), (64, 3)), capfd=None):
    """Every exact / SQL statement on `idx` (with deletions) against `twin` (the live rows only) and the oracle."""
    live = np.flatnonzero(~dead)
    xl, rl = x[live], rid[live]
    for op, oop in ((VectorOp.L2Distance, ob.L2), (VectorOp.CosineDistance, ob.COSINE)):
        for limit, offset in grid:
            for proj in (None, VectorOp.InnerProduct):
                a, b = VectorScanBatch(idx, op, limit, offset, project=proj), VectorScanBatch(twin, op, limit, offset, project=proj)
                got, want = a.execute(q), b.execute(q)
                for g_, w_ in zip(got, want):
                    same_bits(g_, w_, ("sql_topk", op, limit, offset))
                if proj is not None:
                    same_bits(a.projected, b.projected)
            if (limit, offset) == (64, 3) and len(live):
                o_rows, o_keys, o_counts = ob.sql_topk(xl, q, 64, oop, 3, n_threads=8)
                assert np.array_equal(got[2], o_counts)
                have = o_rows != INVALID_ROW
                assert np.array_equal(got[0][have], rl[o_rows[have].astype(np.int64)])
                same_bits(got[1][have], o_keys[have])
    for metric in (DistanceFunction.L2, DistanceFunction.Cosine, DistanceFunction.InnerProduct):
        got, want = idx.bruteforce_topk(q, 10, metric), twin.bruteforce_topk(q, 10, metric)
        same_bits(got[0], want[0])
        same_bits(got[2], want[2])
        same_bits(got[3], want[3])
        nodes = np.where(want[1] == 0xFFFFFFFF, 0xFFFFFFFF, live[np.minimum(want[1], len(live) - 1)] if len(live) else 0)
        assert np.array_equal(got[1], nodes.astype(np.uint32))
    for op, cmp in NEAR:
        sign = -1.0 if op == VectorOp.InnerProduct else 1.0  # the near direction first
        radii = sign * np.sort(sign * approx_values(x, q, op), axis=1)[:, min(60, x.shape[0] - 1)]
        for limit, offset in ((0, 0), (10, 0), (7, 5)):
            got = VectorRangeScanBatch(idx, op, cmp, limit, offset).execute(q, radii)
            want = VectorRangeScanBatch(twin, op, cmp, limit, offset).execute(q, radii)
            for g_, w_ in zip(got, want):
                same_bits(g_, w_, ("sql_range", op, cmp, limit, offset))
        for order in (VectorOp.L2Distance, VectorOp.CosineDistance):
            got = VectorRangeTopKBatch(idx, op, cmp, order, 10, 2).execute(q, radii)
            want = VectorRangeTopKBatch(twin, op, cmp, order, 10, 2).execute(q, radii)
            for g_, w_ in zip(got, want):
                same_bits(g_, w_, ("sql_range_topk", op, cmp, order))


@pytest.mark.parametrize("frac", [0.01, 0.1, 0.5, 1.0])
def test_sql_and_exact_equal_the_live_table(gpu_required, frac):
    x = ds.gaussian_latent(20_000, 96, seed=61)
    q = ds.gaussian_latent(48, 96, seed=62)
    rid = np.arange(20_000, dtype=np.uint64) * 2 + 1
    dead = deleted_mask(20_000, frac, 63)
    idx, twin = table_index(x, rid), table_index(x[~dead], rid[~dead])
    idx.delete(np.flatnonzero(dead))
    compare_statements(idx, twin, x, rid, dead, q)
    idx.close()
    twin.close()


def test_use_index_is_topk_over_the_filtered_traversal(gpu_required, small_graph):
    g, arrays = small_graph
    dead = deleted_mask(g.n, 0.3, 65)
    q = ds.gaussian_latent(16, 128, seed=66)
    idx, twin = CudaHnswIndex.from_graph(arrays), CudaHnswIndex.from_graph(arrays)
    idx.delete(np.flatnonzero(dead))
    for op, oop in ((VectorOp.L2Distance, ob.L2), (VectorOp.CosineDistance, ob.COSINE)):
        # the statement's traversal runs with the ORDER BY operator's metric
        _, nodes, _, counts, _ = twin.search_batch(q, 64, 64, DistanceFunction(int(op)), visible=visibility_bitmap(~dead))
        rows, keys, cnt = VectorScanBatch(idx, op, 10, 0, use_index=True, ef_search=64).execute(q)
        for i in range(len(q)):
            scan = np.sort(nodes[i, :counts[i]])  # TopKExec over the rows the traversal returns, in scan order
            o_rows, o_keys, o_cnt = ob.sql_topk(arrays["vectors"][scan], q[i], 10, oop)
            assert cnt[i] == o_cnt[0]
            assert np.array_equal(rows[i, :cnt[i]], arrays["row_ids"][scan[o_rows[0, :cnt[i]].astype(np.int64)]])
            same_bits(keys[i, :cnt[i]], o_keys[0, :cnt[i]])
    idx.close()
    twin.close()


def test_ties_and_mass_duplicates(gpu_required):
    rng = np.random.default_rng(71)
    base = ds.gaussian_latent(500, 48, seed=72)
    x = np.repeat(base, 20, axis=0)                   # every row 20 times: ties at every key
    x[:3000] = base[0]                                # and 3000 copies of one row
    rid = rng.permutation(10_000).astype(np.uint64)
    dead = rng.random(10_000) < 0.3
    dead[:3000:2] = True                              # deleted rows among the mass duplicates
    q = np.concatenate([base[:24], ds.gaussian_latent(24, 48, seed=73)])
    idx, twin = table_index(x, rid), table_index(x[~dead], rid[~dead])
    idx.delete(np.flatnonzero(dead))
    compare_statements(idx, twin, x, rid, dead, q, grid=((10, 0), (64, 3), (500, 12)))
    idx.close()
    twin.close()


def test_nearest_rows_of_every_query_deleted(gpu_required, capfd, monkeypatch):
    """K deleted near-duplicates of a query must not raise the filter's threshold above the live rows of the result."""
    x = ds.gaussian_latent(20_000, 96, seed=81)
    q = x[np.random.default_rng(82).choice(20_000, 64, replace=False)] + 1e-3
    d = approx_values(x, q, VectorOp.L2Distance)
    dead = np.zeros(20_000, bool)
    dead[np.argsort(d, axis=1)[:, :50].ravel()] = True
    rid = np.arange(20_000, dtype=np.uint64)
    idx, twin = table_index(x, rid), table_index(x[~dead], rid[~dead])
    idx.delete(np.flatnonzero(dead))
    monkeypatch.setenv("TURDB_EXACT_VERBOSE", "1")
    for op, oop in ((VectorOp.L2Distance, ob.L2), (VectorOp.CosineDistance, ob.COSINE)):
        got = VectorScanBatch(idx, op, 10).execute(q)
        assert fallbacks(capfd, "topk") == 0
        for g_, w_ in zip(got, VectorScanBatch(twin, op, 10).execute(q)):
            same_bits(g_, w_)
        o_rows, o_keys, o_counts = ob.sql_topk(x[~dead], q, 10, oop, n_threads=8)
        assert np.array_equal(got[0], rid[~dead][o_rows.astype(np.int64)]) and np.array_equal(got[2], o_counts)
        same_bits(got[1], o_keys)
    for metric in (DistanceFunction.L2, DistanceFunction.Cosine):
        got, want = idx.bruteforce_topk(q, 10, metric), twin.bruteforce_topk(q, 10, metric)
        same_bits(got[0], want[0])
        same_bits(got[2], want[2])
    idx.close()
    twin.close()


@pytest.mark.parametrize("dim,force_bf16", [(37, False), (96, True), (131, True)])
def test_odd_dims_and_forced_bf16(gpu_required, monkeypatch, dim, force_bf16):
    if force_bf16:
        monkeypatch.setenv("TURDB_EXACT_FORCE_BF16", "1")
    x = ds.gaussian_latent(6000, dim, seed=dim)
    q = ds.gaussian_latent(32, dim, seed=dim + 1)
    rid = np.arange(6000, dtype=np.uint64) + 7
    dead = deleted_mask(6000, 0.1, dim)
    idx, twin = table_index(x, rid), table_index(x[~dead], rid[~dead])
    idx.delete(np.flatnonzero(dead))
    compare_statements(idx, twin, x, rid, dead, q, grid=((10, 0), (64, 3)))
    idx.close()
    twin.close()


def test_delete_before_and_after_the_copies_and_after_insert(gpu_required):
    x = ds.gaussian_latent(8000, 64, seed=91)
    q = ds.gaussian_latent(32, 64, seed=92)
    rid = np.arange(8000, dtype=np.uint64) * 5
    rnd = 1.0 - np.random.default_rng(93).random(8000)
    d1, d2 = deleted_mask(6000, 0.05, 94), deleted_mask(6000, 0.05, 95)
    idx = CudaHnswIndex.build(x[:6000], rid[:6000], rnd[:6000], max_batch=256)
    idx.delete(np.flatnonzero(d1))                    # before the 16-bit copies exist
    dead = d1.copy()
    compare_statements(idx, table_index(x[:6000][~dead], rid[:6000][~dead]), x[:6000], rid[:6000], dead, q, grid=((10, 0),))
    idx.delete(np.flatnonzero(d2))                    # after
    dead |= d2
    compare_statements(idx, table_index(x[:6000][~dead], rid[:6000][~dead]), x[:6000], rid[:6000], dead, q, grid=((10, 0),))
    idx.insert(x[6000:], rid[6000:], rnd[6000:])      # drops the copies (and grows the index)
    dead = np.concatenate([dead, np.zeros(2000, bool)])
    compare_statements(idx, table_index(x[~dead], rid[~dead]), x, rid, dead, q, grid=((10, 0), (64, 3)))
    idx.close()


# ---- 5. deleting does not move statements to the streaming scan ----------------------------------------------------
def test_no_new_fallback(gpu_required, capfd, monkeypatch):
    x = ds.gaussian_latent(20_000, 96, seed=101)
    q = ds.gaussian_latent(64, 96, seed=102)
    idx, plain = table_index(x), table_index(x)
    idx.delete(np.flatnonzero(deleted_mask(20_000, 0.01, 103)))
    monkeypatch.setenv("TURDB_EXACT_VERBOSE", "1")
    for op in (VectorOp.L2Distance, VectorOp.CosineDistance):
        for limit, offset in ((10, 0), (64, 3)):
            VectorScanBatch(plain, op, limit, offset).execute(q)
            base = fallbacks(capfd, "topk")
            VectorScanBatch(idx, op, limit, offset).execute(q)
            assert base == 0 and fallbacks(capfd, "topk") == 0
    idx.close()
    plain.close()


# ---- 6. insert ignores deletions -------------------------------------------------------------------------------------
@pytest.mark.parametrize("n0,n1", [(3000, 400), (2400, 3000)])
def test_insert_after_delete_gives_the_graph_without_deletions(gpu_required, n0, n1):
    """Two inserts per index: the first grows the arrays (a build leaves no spare capacity), the second (n1 = 400) fits
    in place.  A delete between them hits one of the rows the first insert added."""
    x = ds.gaussian_latent(n0 + n1, 32, seed=n0)
    rid = np.arange(n0 + n1, dtype=np.uint64) + 11
    rnd = 1.0 - np.random.default_rng(n1).random(n0 + n1)
    h = n0 + n1 // 2
    idx = CudaHnswIndex.build(x[:n0], rid[:n0], rnd[:n0], max_batch=64)
    twin = CudaHnswIndex.build(x[:n0], rid[:n0], rnd[:n0], max_batch=64)
    dead = np.zeros(n0 + n1, bool)
    dead[:n0] = deleted_mask(n0, 0.2, 3)
    assert idx.delete(np.flatnonzero(dead)) == int(dead.sum())
    for lo, hi in ((n0, h), (h, n0 + n1)):
        idx.insert(x[lo:hi], rid[lo:hi], rnd[lo:hi], max_batch=64)
        twin.insert(x[lo:hi], rid[lo:hi], rnd[lo:hi], max_batch=64)
        if lo == n0:
            dead[[n0, n0 + 5, 17]] = True
            assert idx.delete([n0, n0 + 5, 17]) == int(dead.sum())
    a, b = idx.export_graph(), twin.export_graph()
    assert a["entry"] == b["entry"] and a["max_level"] == b["max_level"]
    for key in GRAPH_KEYS:
        assert np.array_equal(a[key], b[key]), key
    assert idx.delete([]) == int(dead.sum())  # deleted nodes stay deleted, new rows are live
    q = x[h:h + 32]
    rows = idx.bruteforce_topk(q, 1)[0]
    assert np.array_equal(rows[:, 0], rid[h:h + 32])
    got = idx.search_batch(x[n0 - 16:n0 + 16], 10, 64)
    same_traversal(got, twin.search_batch(x[n0 - 16:n0 + 16], 10, 64, visible=visibility_bitmap(~dead)))
    live_twin = table_index(x[~dead], rid[~dead])
    for g_, w_ in zip(VectorScanBatch(idx, VectorOp.L2Distance, 10).execute(x[n0 - 16:n0 + 16]),
                      VectorScanBatch(live_twin, VectorOp.L2Distance, 10).execute(x[n0 - 16:n0 + 16])):
        same_bits(g_, w_)
    for ix in (idx, twin, live_twin):
        ix.close()


# ---- 7. errors and counts ----------------------------------------------------------------------------------------------
def test_invalid_ids_change_nothing_and_counts_stay_exact(gpu_required):
    x = ds.gaussian_latent(5000, 32, seed=111)
    q = ds.gaussian_latent(16, 32, seed=112)
    idx = table_index(x)
    nbytes = idx.info()["device_bytes"]
    L = _lib.load()
    out = C.c_uint64(99)
    bad = np.array([1, 5000, 2], np.uint32)
    assert L.turdb_cuda_index_delete(idx._h, 3, bad.ctypes.data_as(C.POINTER(C.c_uint32)), C.byref(out)) == _lib.ERR_INVALID_ARGUMENT
    assert b"5000" in L.turdb_cuda_last_error() and out.value == 99
    assert idx.delete([]) == 0 and idx.info()["device_bytes"] == nbytes  # nothing allocated, nothing deleted
    assert idx.delete([1, 2, 2]) == 2
    assert idx.info()["device_bytes"] == nbytes + (5000 + 63) // 64 * 8
    before = VectorScanBatch(idx, VectorOp.L2Distance, 10).execute(q)
    assert L.turdb_cuda_index_delete(idx._h, 3, bad.ctypes.data_as(C.POINTER(C.c_uint32)), None) == _lib.ERR_INVALID_ARGUMENT
    for g_, w_ in zip(VectorScanBatch(idx, VectorOp.L2Distance, 10).execute(q), before):
        same_bits(g_, w_)
    assert idx.delete([2, 3]) == 3 and idx.delete([3, 3, 1]) == 3 and idx.delete([]) == 3
    assert idx.delete(np.arange(5000)) == 5000
    rows, keys, counts = VectorScanBatch(idx, VectorOp.L2Distance, 10).execute(q)
    assert (counts == 0).all() and (rows == INVALID_ROW).all()
    idx.close()
