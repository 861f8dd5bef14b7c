"""Appending rows to a resident index (turdb_cuda_index_insert, csrc/graph_insert.inl): the insert path continued from
the current node count must give the graph one build over all rows gives — the oracle's graph with max_batch = 1, the
device build's own graph, array for array, when the split falls on a step boundary — for built, uploaded, file-read and
empty indexes; derived arenas (norms, SQ8 rows, the exact path's 16-bit copies) must answer for the new rows; growth
copies the index O(log n) times; a rejected call leaves the index as it was."""
import ctypes as C

import numpy as np
import pytest

from oracle import binding as ob
from test_gpu_build import graphs_equal
from turdb_b200 import _lib
from turdb_b200 import datasets as ds
from turdb_b200.hnsw import CudaHnswIndex, DistanceFunction
from turdb_b200.hnsw_file import HnswFile
from turdb_b200.sql_operator import VectorOp, VectorScanBatch

pytestmark = pytest.mark.gpu

KEYS = ("vectors", "row_ids", "levels", "l0_adj", "l0_cnt", "up_base", "up_adj", "up_cnt")


def same_graph(a, b):
    assert a["entry"] == b["entry"] and a["max_level"] == b["max_level"]
    for key in KEYS:
        assert np.array_equal(a[key], b[key]), key


def same_search(a, b, q, ef=64):
    ra, rb = a.search_batch(q, 10, ef, DistanceFunction.L2), b.search_batch(q, 10, ef, DistanceFunction.L2)
    assert np.array_equal(ra[0], rb[0]) and np.array_equal(ra[2].view(np.uint32), rb[2].view(np.uint32))
    assert np.array_equal(ra[3], rb[3]) and np.array_equal(ra[4], rb[4])


def corpus(n, dim, seed):
    return ds.gaussian_latent(n, dim, seed=seed), np.arange(n, dtype=np.uint64) * 3 + 1, ob.level_randoms(n, seed + 1)


def schedule(n, max_batch):
    """First node of every step of a build over n nodes (graph_insert.inl): node 0 alone, then steps of
    min(max_batch, max(1, s // 8), n - s)."""
    starts, s = [], 1
    while s < n:
        starts.append(s)
        s += min(max_batch, max(1, s // 8), n - s)
    return starts


@pytest.mark.parametrize("n,dim,mode,k", [(3000, 32, ob.BUILD_INTENT, 2000), (3000, 32, ob.BUILD_VERBATIM, 2000),
                                          (1200, 384, ob.BUILD_INTENT, 800)])
def test_sequential_append_equals_the_oracle(gpu_required, n, dim, mode, k):
    x, rid, rnd = corpus(n, dim, n + dim)
    og = ob.OracleGraph.new(dim, 16, 100, mode)
    og.insert_batch(rid, x, rnd)
    full = CudaHnswIndex.build(x, rid, rnd, m=16, ef_construction=100, mode=mode, max_batch=1)
    one = CudaHnswIndex.build(x[:k], rid[:k], rnd[:k], m=16, ef_construction=100, mode=mode, max_batch=1)
    one.insert(x[k:], rid[k:], rnd[k:], max_batch=1)
    assert one.n == n and one.info()["n"] == n
    many = CudaHnswIndex.build(x[:k], rid[:k], rnd[:k], m=16, ef_construction=100, mode=mode, max_batch=1)
    cuts = [k, k + 1, k + 2, k + 9, k + 10, k + 137, k + 138, (k + n) // 2, n - 1, n]
    for a, b in zip(cuts[:-1], cuts[1:]):
        many.insert(x[a:b], rid[a:b], rnd[a:b], max_batch=1)
    g = one.export_graph()
    graphs_equal(g, og.export(), x)
    same_graph(g, full.export_graph())
    same_graph(many.export_graph(), g)
    q = ds.gaussian_latent(50, dim, seed=5)
    gpu = one.search_batch(q, 10, 64, DistanceFunction.L2)
    cpu = ob.OracleGraph.from_arrays(g).search(q, 10, 64, ob.L2)
    assert np.array_equal(gpu[1], cpu[1]) and np.array_equal(gpu[2].view(np.uint32), cpu[2].view(np.uint32))
    for i in (full, one, many):
        i.close()


def test_batched_append_at_step_boundaries_equals_batched_build(gpu_required):
    n, dim, mb = 20000, 64, 1024
    x, rid, rnd = corpus(n, dim, 7)
    starts = schedule(n, mb)
    b1 = next(s for s in starts if s >= 9000)
    b2 = next(s for s in starts if s >= 15000)
    full = CudaHnswIndex.build(x, rid, rnd, max_batch=mb)
    idx = CudaHnswIndex.build(x[:b1], rid[:b1], rnd[:b1], max_batch=mb)
    idx.insert(x[b1:b2], rid[b1:b2], rnd[b1:b2], max_batch=mb)
    idx.insert(x[b2:], rid[b2:], rnd[b2:], max_batch=mb)
    same_graph(idx.export_graph(), full.export_graph())
    same_search(idx, full, ds.gaussian_latent(100, dim, seed=8))
    idx.close()
    full.close()


def test_batched_append_off_boundary_keeps_quality(gpu_required):
    n, dim, mb = 20000, 64, 1024
    x, rid, rnd = corpus(n, dim, 9)
    split = 12345
    assert split not in schedule(n, mb)
    q = ds.gaussian_latent(300, dim, seed=2)
    og = ob.OracleGraph.new(dim, 16, 100, ob.BUILD_INTENT)
    og.insert_batch(rid, x, rnd)
    d = ((q[:, None, :] - x[None, :, :]) ** 2).sum(-1)
    gt = rid[np.argsort(d, axis=1, kind="stable")[:, :10]]

    def recall(rows):
        return float(np.mean([len(set(rows[i].tolist()) & set(gt[i].tolist())) / 10 for i in range(len(q))]))
    seq = og.search(q, 10, 64, ob.L2, n_threads=8)
    idx = CudaHnswIndex.build(x[:split], rid[:split], rnd[:split], max_batch=mb)
    idx.insert(x[split:], rid[split:], rnd[split:], max_batch=mb)
    g = idx.export_graph()
    assert (g["l0_cnt"] > 0).all(), "every node is linked"
    bat = idx.search_batch(q, 10, 64, DistanceFunction.L2)
    assert recall(bat[0]) >= recall(seq[0]) - 0.02, (recall(bat[0]), recall(seq[0]))
    cpu = ob.OracleGraph.from_arrays(g).search(q, 10, 64, ob.L2, n_threads=8)
    assert np.array_equal(bat[1], cpu[1]) and np.array_equal(bat[2].view(np.uint32), cpu[2].view(np.uint32))
    idx.close()


def test_uploaded_graph_grows_like_the_oracle(gpu_required):
    n, dim, k = 3000, 32, 2000
    x, rid, rnd = corpus(n, dim, 21)
    og = ob.OracleGraph.new(dim, 16, 100, ob.BUILD_INTENT)
    og.insert_batch(rid[:k], x[:k], rnd[:k])
    up = CudaHnswIndex.from_graph(og.export())
    with pytest.raises(ValueError, match="required"):
        up.insert(x[k:], rid[k:], rnd[k:])  # from_graph knows no build parameters
    up.insert(x[k:], rid[k:], rnd[k:], m=16, ef_construction=100, mode=ob.BUILD_INTENT, max_batch=1)
    # the same graph written as a .hnsw file (dense ids follow the file's node order), uploaded, grown with the header's
    # M / ef_construction
    data, _, _ = ob.hnsw_file_write(og, mode=1)
    f = HnswFile.from_bytes(data)
    assert (f.info["m"], f.info["ef_construction"]) == (16, 100)
    fi = f.upload(vectors=x[:k])
    fi.insert(x[k:], rid[k:], rnd[k:], max_batch=1)
    og.insert_batch(rid[k:], x[k:], rnd[k:])
    o = og.export()
    graphs_equal(up.export_graph(), o, x)
    graphs_equal(fi.export_graph(), o, x)
    q = ds.gaussian_latent(50, dim, seed=5)
    gpu = fi.search_batch(q, 10, 64, DistanceFunction.L2)
    cpu = ob.OracleGraph.from_arrays(fi.export_graph()).search(q, 10, 64, ob.L2)
    assert np.array_equal(gpu[0], cpu[0]) and np.array_equal(gpu[2].view(np.uint32), cpu[2].view(np.uint32))
    for i in (up, fi):
        i.close()
    f.close()


def test_empty_index_grows_like_build(gpu_required):
    n, dim = 1500, 24
    x, rid, rnd = corpus(n, dim, 31)
    ref = CudaHnswIndex.build(x, rid, rnd, max_batch=64).export_graph()
    built = CudaHnswIndex.build(np.zeros((0, dim), np.float32), max_batch=64)
    assert built.info()["entry"] is None
    built.insert(x[:1], rid[:1], rnd[:1], max_batch=64)  # the first row only becomes the entry
    built.insert(x[1:], rid[1:], rnd[1:], max_batch=64)
    same_graph(built.export_graph(), ref)
    empty = dict(vectors=np.zeros((0, dim), np.float32), row_ids=np.zeros(0, np.uint64), levels=np.zeros(0, np.uint8),
                 l0_adj=np.zeros((0, 32), np.uint32), l0_cnt=np.zeros(0, np.uint8), up_base=np.zeros(0, np.uint32),
                 up_adj=np.zeros((0, 16), np.uint32), up_cnt=np.zeros(0, np.uint8), entry=0, max_level=0)
    up = CudaHnswIndex.from_graph(empty)
    up.insert(x, rid, rnd, m=16, ef_construction=100, mode=1, max_batch=64)
    same_graph(up.export_graph(), ref)
    built.close()
    up.close()


def test_appended_node_above_max_level_becomes_the_entry(gpu_required):
    x = ds.gaussian_latent(30, 16, seed=3)
    rnd = np.full(30, 0.9)
    rnd[0] = 0.05   # level 1
    rnd[20] = 1e-4  # level 3 > max_level 1: appended, it becomes the entry with a one-way upper link
    rid = np.arange(30, dtype=np.uint64)
    og = ob.OracleGraph.new(16, 16, 100, ob.BUILD_INTENT)
    og.insert_batch(rid, x, rnd)
    idx = CudaHnswIndex.build(x[:20], rid[:20], rnd[:20], max_batch=1)
    assert idx.info()["max_level"] == 1
    idx.insert(x[20:], rid[20:], rnd[20:], max_batch=1)
    g = idx.export_graph()
    graphs_equal(g, og.export(), x)
    assert g["entry"] == 20 and g["max_level"] == 3 and idx.info()["entry"] == 20
    idx.close()


def test_sq8_rows_follow_an_insert(gpu_required):
    from test_gpu_sq8 import run_sq8
    n, dim, k = 3000, 48, 2000
    x, rid, rnd = corpus(n, dim, 41)
    idx = CudaHnswIndex.build(x[:k], rid[:k], rnd[:k], max_batch=256)
    idx.enable_sq8()
    idx.insert(x[k:], rid[k:], rnd[k:], max_batch=256)
    fresh = CudaHnswIndex.from_graph(idx.export_graph())
    fresh.enable_sq8()
    q = ds.gaussian_latent(200, dim, seed=6)
    for metric in (ob.L2, ob.COSINE, ob.IP):
        a, b = run_sq8(idx, q, 10, 64, metric), run_sq8(fresh, q, 10, 64, metric)
        assert np.array_equal(a[3], b[3]) and np.array_equal(a[1], b[1]) and np.array_equal(a[0], b[0])
        assert np.array_equal(a[2].view(np.uint32), b[2].view(np.uint32)) and np.array_equal(a[4], b[4])
    idx.close()
    fresh.close()


def test_exact_path_and_sql_operator_see_appended_rows(gpu_required):
    n, dim, k = 4000, 96, 3000
    x, rid, rnd = corpus(n, dim, 51)
    x[-1] *= 1e3  # a new row far larger than every old one: stale 16-bit copies would keep the old format and scale
    idx = CudaHnswIndex.build(x[:k], rid[:k], rnd[:k], max_batch=256)
    q = ds.gaussian_latent(64, dim, seed=7)
    for metric in DistanceFunction:
        idx.bruteforce_topk(q, 10, metric)  # builds the copies of the first k rows
    VectorScanBatch(idx, VectorOp.L2Distance, 10).execute(q)
    idx.insert(x[k:], rid[k:], rnd[k:], max_batch=256)
    fresh = CudaHnswIndex.from_graph(idx.export_graph())
    for metric in DistanceFunction:
        a, b = idx.bruteforce_topk(q, 10, metric), fresh.bruteforce_topk(q, 10, metric)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[2].view(np.uint32), b[2].view(np.uint32)), metric
        assert np.array_equal(a[3], b[3])
    for op in (VectorOp.L2Distance, VectorOp.CosineDistance):
        a, b = VectorScanBatch(idx, op, 10).execute(q), VectorScanBatch(fresh, op, 10).execute(q)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1].view(np.uint64), b[1].view(np.uint64)), op
        assert np.array_equal(a[2], b[2])
    o_rows, o_keys, _ = ob.sql_topk(x, q, 10, op=ob.L2, n_threads=4)  # oracle rows = positions in x
    a = VectorScanBatch(idx, VectorOp.L2Distance, 10).execute(q)
    assert np.array_equal(a[0], rid[o_rows.astype(np.int64)]) and np.array_equal(a[1].view(np.uint64), o_keys.view(np.uint64))
    idx.close()
    fresh.close()


def test_single_row_inserts_grow_geometrically(gpu_required):
    n, dim, k = 10200, 16, 10000
    x, rid, rnd = corpus(n, dim, 61)
    full = CudaHnswIndex.build(x, rid, rnd, max_batch=1)
    idx = CudaHnswIndex.build(x[:k], rid[:k], rnd[:k], max_batch=1)
    sizes = [idx.info()["device_bytes"]]
    for i in range(k, n):
        idx.insert(x[i:i + 1], rid[i:i + 1], rnd[i:i + 1])
        sizes.append(idx.info()["device_bytes"])
    changes = int(np.count_nonzero(np.diff(sizes)))
    assert 1 <= changes <= 3, changes  # one growth of the node arrays (x1.5 > 200 rows), at most two of the slot arrays
    assert idx.info()["n"] == n
    same_graph(idx.export_graph(), full.export_graph())
    same_search(idx, full, ds.gaussian_latent(100, dim, seed=62))
    idx.close()
    full.close()


def test_rejected_insert_leaves_the_index_unchanged(gpu_required):
    n, dim = 3000, 32
    x, rid, rnd = corpus(n, dim, 71)
    idx = CudaHnswIndex.build(x, rid, rnd, max_batch=256)
    q = ds.gaussian_latent(50, dim, seed=72)
    info0, g0, s0 = idx.info(), idx.export_graph(), idx.search_batch(q, 10, 64)
    L = _lib.load()
    wide = ds.gaussian_latent(4, dim + 1, seed=73)
    v = np.ascontiguousarray(wide[:, :dim])
    r = np.arange(4, dtype=np.uint64) + 10**6
    u = np.full(4, 0.5)

    def call(bp, vec=v, rows=r):
        return L.turdb_cuda_index_insert(idx._h, C.byref(bp), 4, None if vec is None else vec.ctypes.data_as(C.POINTER(C.c_float)),
                                         None if rows is None else rows.ctypes.data_as(C.POINTER(C.c_uint64)),
                                         u.ctypes.data_as(C.POINTER(C.c_double)))
    assert call(_lib.BuildParams(dim + 1, 16, 100, 1, 64, 0), wide) == _lib.ERR_DIMENSION_MISMATCH
    assert b"does not match index dimension" in L.turdb_cuda_last_error()
    assert call(_lib.BuildParams(dim, 1, 100, 1, 64, 0)) == _lib.ERR_UNSUPPORTED
    assert call(_lib.BuildParams(dim, 16, 0, 1, 64, 0)) == _lib.ERR_INVALID_ARGUMENT
    assert call(_lib.BuildParams(dim, 16, 100, 1, 64, 0), vec=None) == _lib.ERR_INVALID_ARGUMENT
    assert call(_lib.BuildParams(dim, 16, 100, 1, 64, 0), rows=None) == _lib.ERR_INVALID_ARGUMENT
    assert L.turdb_cuda_index_insert(idx._h, None, 4, None, None, None) == _lib.ERR_INVALID_ARGUMENT
    with pytest.raises(ValueError):
        idx.insert(wide, r, u)
    idx.insert(v[:0], r[:0], u[:0])  # n == 0: a no-op
    assert idx.info() == info0 and idx.n == n
    same_graph(idx.export_graph(), g0)
    s1 = idx.search_batch(q, 10, 64)
    assert all(np.array_equal(a, b) for a, b in zip(s0, s1))
    # and the index still takes rows afterwards
    idx.insert(v, r, u)
    assert idx.info()["n"] == n + 4
    idx.close()
