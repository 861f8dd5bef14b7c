"""Compacting a resident index (turdb_cuda_index_compact): the device's graph must equal the CPU reference's compaction
(tests/compact_reference.py) of the same graph array for array; traversals must equal the oracle's search on it; every
exact statement must answer bit for bit as before the call and as an index of the live rows; SQ8, insert, `.hnsw`
uploads with tombstones and the no-op case follow."""
import struct

import numpy as np
import pytest
import torch

import compact_reference
from oracle import binding as ob
from turdb_b200 import datasets as ds
from turdb_b200.hnsw import INVALID_NODE, CudaHnswIndex, DistanceFunction
from turdb_b200.hnsw_file import HnswFile
from turdb_b200.sql_operator import RangeCmp, VectorOp, VectorRangeScanBatch, VectorRangeTopKBatch, VectorScanBatch

pytestmark = pytest.mark.gpu

GRAPH_KEYS = ("vectors", "row_ids", "levels", "l0_adj", "l0_cnt", "up_base", "up_adj", "up_cnt")


def table_index(x, row_ids):
    n = x.shape[0]
    g = dict(vectors=x, row_ids=row_ids, levels=np.zeros(n, np.uint8), l0_adj=np.full((n, 32), INVALID_NODE, np.uint32),
             l0_cnt=np.zeros(n, np.uint8), up_base=np.full(n, INVALID_NODE, np.uint32), up_adj=np.zeros((0, 16), np.uint32),
             up_cnt=np.zeros(0, np.uint8), entry=0 if n else INVALID_NODE, max_level=0)
    return CudaHnswIndex.from_graph(g)


def deleted_mask(n, frac, seed):
    return np.random.default_rng(seed).random(n) < frac if frac < 1.0 else np.ones(n, bool)


def same_bits(a, b, what=""):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    assert a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8)), what


def same_graph(got, want):
    for key in GRAPH_KEYS:
        same_bits(got[key], want[key], key)
    assert (got["entry"], got["max_level"]) == (want["entry"], want["max_level"])


def same_as_oracle(got, cpu):
    assert np.array_equal(got[3], cpu[3]), "counts differ"
    for i in range(len(got[3])):
        c = cpu[3][i]
        assert np.array_equal(got[1][i][:c], cpu[1][i][:c]), i
        assert np.array_equal(got[2][i][:c].view(np.uint32), cpu[2][i][:c].view(np.uint32)), i
    for f in ("n_dist", "n_expanded"):
        assert np.array_equal(got[4][f], cpu[4][f]), f


def compact_both(idx, arrays, dead):
    """Delete `dead` on the device index and compact it; the CPU reference compacts the same graph.  Returns (map, the
    oracle graph of the reference's result)."""
    assert idx.delete(np.flatnonzero(dead)) == int(dead.sum())
    o2n = idx.compact()
    ref, ref_o2n = compact_reference.compact(arrays, ~dead)
    og = ob.OracleGraph.from_arrays(ref)
    assert np.array_equal(ref_o2n, o2n)
    prefix = np.cumsum(~dead) - 1
    assert np.array_equal(o2n, np.where(dead, INVALID_NODE, prefix).astype(np.uint32))
    assert idx.n == og.n == int((~dead).sum())
    return o2n, og


# ---- 1. the graph equals the reference's compaction, the traversals the oracle's search on it -----------------------
@pytest.mark.parametrize("frac", [0.0, 0.01, 0.1, 0.5, 1.0])
@pytest.mark.parametrize("entry_deleted", [False, True])
def test_graph_and_traversals_equal_the_oracle(gpu_required, small_graph, frac, entry_deleted):
    g, arrays = small_graph
    dead = deleted_mask(g.n, frac, int(frac * 1000) + 11)
    dead[arrays["entry"]] = entry_deleted or frac == 1.0
    idx = CudaHnswIndex.from_graph(arrays)
    before = idx.info()["device_bytes"]
    _, og = compact_both(idx, arrays, dead)
    got = idx.export_graph()
    same_graph(got, og.export())
    assert idx.delete([]) == 0
    info = idx.info()
    live = int((~dead).sum())
    assert info["n"] == live
    # the deleted rows' share of the arena (128 floats) and of the level-0 adjacency leaves the device
    assert before - info["device_bytes"] >= int(dead.sum()) * (128 * 4 + 32 * 4)
    q = ds.gaussian_latent(64, 128, seed=91)
    for form in (1, 2):
        idx.set_traversal_form(form)
        for metric in (ob.L2, ob.COSINE, ob.IP):
            res = idx.search_batch(q, 10, 64, DistanceFunction(metric))
            if live == 0:
                assert (res[3] == 0).all()
                continue
            same_as_oracle(res, og.search(q, 10, 64, metric, n_threads=8))
            assert (res[1][res[1] != INVALID_NODE] < live).all()
    idx.close()


# ---- 2. exact statements answer as before the call and as the live rows --------------------------------------------
def statements(idx, q):
    out = []
    for op in (VectorOp.L2Distance, VectorOp.CosineDistance):
        for limit, offset in ((10, 0), (5, 7), (64, 3)):
            out += list(VectorScanBatch(idx, op, limit, offset).execute(q))
    for metric in (DistanceFunction.L2, DistanceFunction.Cosine, DistanceFunction.InnerProduct):
        rows, nodes, dist, counts = idx.bruteforce_topk(q, 10, metric)
        out += [rows, dist, counts]
    for op, cmp in ((VectorOp.L2Distance, RangeCmp.Lt), (VectorOp.CosineDistance, RangeCmp.Le),
                    (VectorOp.InnerProduct, RangeCmp.Gt)):
        radius = {VectorOp.L2Distance: 1.1, VectorOp.CosineDistance: 0.6, VectorOp.InnerProduct: 0.4}[op]
        radii = np.full(len(q), radius)
        for limit, offset in ((0, 0), (7, 5)):
            out += list(VectorRangeScanBatch(idx, op, cmp, limit, offset).execute(q, radii))
        out += list(VectorRangeTopKBatch(idx, op, cmp, VectorOp.L2Distance, 10, 2).execute(q, radii))
    return out


@pytest.mark.parametrize("frac", [0.01, 0.1, 0.5])
def test_exact_statements_unchanged(gpu_required, frac):
    x = ds.gaussian_latent(20_000, 96, seed=61)
    q = ds.gaussian_latent(48, 96, seed=62)
    rid = np.arange(20_000, dtype=np.uint64) * 2 + 1
    dead = deleted_mask(20_000, frac, 63)
    idx, twin = table_index(x, rid), table_index(x[~dead], rid[~dead])
    idx.delete(np.flatnonzero(dead))
    want = statements(twin, q)
    before = statements(idx, q)
    nodes_before = idx.bruteforce_topk(q, 10)[1]
    o2n = idx.compact()
    after = statements(idx, q)
    for i, (a, b, w) in enumerate(zip(after, before, want)):
        same_bits(a, w, ("live table", i))
        same_bits(a, b, ("before the call", i))
    nodes = idx.bruteforce_topk(q, 10)[1]
    mapped = np.where(nodes_before == INVALID_NODE, INVALID_NODE, o2n[np.minimum(nodes_before, len(o2n) - 1)])
    assert np.array_equal(nodes, mapped)
    idx.close()
    twin.close()


def test_use_index_follows_the_new_graph(gpu_required, small_graph):
    g, arrays = small_graph
    dead = deleted_mask(g.n, 0.1, 65)
    q = ds.gaussian_latent(32, 128, seed=66)
    idx = CudaHnswIndex.from_graph(arrays)
    idx.delete(np.flatnonzero(dead))
    idx.compact()
    twin = CudaHnswIndex.from_graph(idx.export_graph())
    for op in (VectorOp.L2Distance, VectorOp.CosineDistance):
        got = VectorScanBatch(idx, op, 10, 0, use_index=True, ef_search=64).execute(q)
        want = VectorScanBatch(twin, op, 10, 0, use_index=True, ef_search=64).execute(q)
        for a, b in zip(got, want):
            same_bits(a, b, op)
    idx.close()
    twin.close()


# ---- 3. SQ8 rows move with their nodes -----------------------------------------------------------------------------------
def test_sq8_rows_and_traversal(gpu_required, small_graph):
    g, arrays = small_graph
    dead = deleted_mask(g.n, 0.2, 67)
    idx = CudaHnswIndex.from_graph(arrays)
    idx.enable_sq8()
    idx.delete(np.flatnonzero(dead))
    idx.compact()
    twin = CudaHnswIndex.from_graph(idx.export_graph())
    for a, b in zip(idx.enable_sq8(return_rows=True), twin.enable_sq8(return_rows=True)):
        same_bits(a, b, "sq8 rows")
    q = torch.from_numpy(ds.gaussian_latent(64, 128, seed=68)).cuda()
    stream = torch.cuda.current_stream().cuda_stream

    def run(ix):
        out = [torch.zeros((64, 10), dtype=torch.int64, device="cuda"), torch.zeros((64, 10), dtype=torch.float32, device="cuda"),
               torch.zeros(64, dtype=torch.int32, device="cuda"), torch.zeros((64, 10), dtype=torch.int32, device="cuda"),
               torch.zeros((64, 4), dtype=torch.int32, device="cuda")]
        ix.search_batch_sq8_device(q.data_ptr(), 64, 10, 64, 0, out[0].data_ptr(), out[1].data_ptr(), out[2].data_ptr(),
                                   d_nodes=out[3].data_ptr(), d_stats=out[4].data_ptr(), stream=stream)
        torch.cuda.synchronize()
        return [t.cpu().numpy() for t in out]

    for a, b in zip(run(idx), run(twin)):
        same_bits(a, b, "sq8 traversal")
    idx.close()
    twin.close()


# ---- 4. insert after compaction, twice -------------------------------------------------------------------------------
def test_insert_after_compaction_matches_the_oracle(gpu_required):
    n0, n1, dim = 2000, 300, 32
    x = ds.gaussian_latent(n0 + 2 * n1, dim, seed=71)
    rid = np.arange(len(x), dtype=np.uint64) * 7 + 3
    rnd = ob.level_randoms(len(x), 72)
    og = ob.OracleGraph.new(dim, 16, 100, ob.BUILD_INTENT)
    og.insert_batch(rid[:n0], x[:n0], rnd[:n0])
    arrays = og.export()
    idx = CudaHnswIndex.from_graph(arrays)
    for step, (lo, hi, frac) in enumerate(((n0, n0 + n1, 0.1), (n0 + n1, n0 + 2 * n1, 0.3))):
        dead = deleted_mask(idx.n, frac, 73 + step)
        dead[arrays["entry"]] = step == 1  # the second round also removes the entry
        _, oc = compact_both(idx, arrays, dead)
        idx.insert(x[lo:hi], rid[lo:hi], rnd[lo:hi], m=16, ef_construction=100, mode=ob.BUILD_INTENT, max_batch=1)
        oc.insert_batch(rid[lo:hi], x[lo:hi], rnd[lo:hi])
        arrays = oc.export()
        same_graph(idx.export_graph(), arrays)
    idx.close()


def test_insert_into_a_fully_compacted_index(gpu_required, small_graph):
    g, arrays = small_graph
    idx = CudaHnswIndex.from_graph(arrays)
    idx.enable_sq8()
    idx.delete(np.arange(g.n))
    assert (idx.compact() == INVALID_NODE).all()
    info = idx.info()
    assert (info["n"], info["entry"], info["max_level"]) == (0, None, 0)
    q = ds.gaussian_latent(8, 128, seed=75)
    assert (idx.search_batch(q, 10, 32)[3] == 0).all() and (idx.bruteforce_topk(q, 10)[3] == 0).all()
    x = ds.gaussian_latent(500, 128, seed=76)
    rid = np.arange(500, dtype=np.uint64)
    rnd = ob.level_randoms(500, 77)
    idx.insert(x, rid, rnd, m=16, ef_construction=100, mode=ob.BUILD_INTENT, max_batch=1)
    og = ob.OracleGraph.new(128, 16, 100, ob.BUILD_INTENT)
    og.insert_batch(rid, x, rnd)
    same_graph(idx.export_graph(), og.export())
    codes, _, _ = idx.enable_sq8(return_rows=True)
    assert np.array_equal(codes, ob.sq8_encode(x)[0])
    idx.close()


# ---- 5. an uploaded .hnsw index: tombstones and absent (+inf) vectors ---------------------------------------------------
def test_uploaded_file_with_tombstones_and_absent_vectors(gpu_required):
    x = ds.gaussian_latent(2000, 32, seed=5)
    g = ob.OracleGraph.build(x, m=16, ef_construction=60, mode=ob.BUILD_INTENT, seed=9,
                             row_ids=np.arange(2000, dtype=np.uint64) * 5 + 11)
    arrays = g.export()
    data, pages, slots = ob.hnsw_file_write(g, mode=1)
    buf = bytearray(data)
    for victim in (50, 900, 1300):  # HnswPage::mark_deleted, storage.rs:671-688: dangling NodeIds -> tombstones
        so = int(pages[victim]) * 16384 + 64 + 4 * int(slots[victim])
        os_, = struct.unpack_from("<H", buf, so)
        struct.pack_into("<H", buf, so, (os_ & 0x1FFF) | (2 << 13))
    f = HnswFile.from_bytes(bytes(buf))
    gone = {int(arrays["row_ids"][i]) for i in (7, 8, 1500, 1501)}
    table = {int(r): x[i] for i, r in enumerate(arrays["row_ids"])}
    idx = f.upload(get_vector=lambda r: None if r in gone else table.get(r))
    ga = idx.export_graph()
    assert np.isinf(ga["vectors"]).all(axis=1).sum() == 7
    dead = deleted_mask(idx.n, 0.3, 78)
    _, og = compact_both(idx, ga, dead)
    got = idx.export_graph()
    same_graph(got, og.export())
    assert np.isinf(got["vectors"]).all(axis=1).sum() == int(np.isinf(ga["vectors"]).all(axis=1)[~dead].sum())
    q = ds.gaussian_latent(100, 32, seed=79)
    for metric in (ob.L2, ob.COSINE, ob.IP):
        same_as_oracle(idx.search_batch(q, 10, 64, DistanceFunction(metric)), og.search(q, 10, 64, metric, n_threads=8))
    idx.close()
    f.close()


# ---- 6. without deletions nothing changes ---------------------------------------------------------------------------------
def test_without_deletions_nothing_changes(gpu_required, small_graph):
    g, arrays = small_graph
    q = ds.gaussian_latent(64, 128, seed=81)
    idx = CudaHnswIndex.from_graph(arrays)

    def answers():
        return (list(idx.search_batch(q, 10, 64)[:4]) + list(idx.bruteforce_topk(q, 10)) +
                list(VectorScanBatch(idx, VectorOp.L2Distance, 10).execute(q)) +
                list(VectorRangeScanBatch(idx, VectorOp.L2Distance, RangeCmp.Lt, 10).execute(q, np.full(64, 9.0))))

    for delete_first in (False, True):
        if delete_first:
            assert idx.delete([]) == 0
        before, nbytes, graph = answers(), idx.info()["device_bytes"], idx.export_graph()
        assert np.array_equal(idx.compact(), np.arange(g.n, dtype=np.uint32))
        assert idx.info()["device_bytes"] == nbytes and idx.n == g.n
        same_graph(idx.export_graph(), graph)
        for a, b in zip(answers(), before):
            same_bits(a, b)
    idx.close()
