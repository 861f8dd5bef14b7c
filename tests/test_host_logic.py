"""Host-side logic that runs without a GPU: datasets, level draws, bitmap packing, the bulk graph builder
(torch on CPU), and the sharded search plumbing under a world_size-2 gloo group."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from oracle import binding as ob
from turdb_b200 import datasets as ds
from turdb_b200.graph_build import build_graph, select_levels
from turdb_b200.hnsw import HnswSearchContext, visibility_bitmap
from turdb_b200.sharding import ShardedSearch, merge_topk_host, shard_bounds


def test_datasets_are_seeded_and_shaped():
    a = ds.gaussian_latent(100, 32, seed=3, normalise=True)
    b = ds.gaussian_latent(100, 32, seed=3, normalise=True)
    assert np.array_equal(a, b) and a.dtype == np.float32
    assert np.allclose(np.linalg.norm(a, axis=1), 1.0, atol=1e-5)
    s = ds.sift_like(50, 128, seed=1)
    assert s.min() >= 0 and s.max() <= 218 and np.array_equal(s, np.rint(s))
    c = ds.clustered(200, 16, seed=2)
    assert c.shape == (200, 16)


def test_select_levels_matches_oracle():
    r = ob.level_randoms(5000, 9)
    lv = select_levels(r, 16)
    ref = np.array([ob.select_level(x, 16) for x in r], np.uint8)
    assert np.array_equal(lv, ref)


def test_visibility_bitmap():
    m = np.zeros(130, bool)
    m[[0, 63, 64, 129]] = True
    w = visibility_bitmap(m)
    assert w.dtype == np.uint64 and w.shape == (3,)
    assert w[0] == (1 | (1 << 63)) and w[1] == 1 and w[2] == 2


def test_search_context_mirrors_reference():
    ctx = HnswSearchContext(32, 1000)
    assert ctx.ef_search() == 32
    ctx.set_ef_search(64)
    assert ctx.ef_search() == 64


def test_bulk_graph_builder_structure_and_recall():
    x = ds.gaussian_latent(3000, 32, seed=1)
    q = ds.gaussian_latent(100, 32, seed=2)
    a = build_graph(x, device="cpu", seed=5, chunk_rows=1024)
    n = len(x)
    assert a["l0_adj"].shape == (n, 32) and a["l0_cnt"].max() <= 32 and a["up_cnt"].max() <= 16
    assert a["levels"][a["entry"]] == a["max_level"]
    for i in range(0, n, 97):  # lists are prefix-packed, in range, without self loops or duplicates
        row = a["l0_adj"][i][:a["l0_cnt"][i]]
        assert (row < n).all() and i not in row and len(set(row.tolist())) == len(row)
        assert (a["l0_adj"][i][a["l0_cnt"][i]:] == 0xFFFFFFFF).all()
    g = ob.OracleGraph.from_arrays(a)
    rows, _, _, _, _ = g.search(q, 10, 64)
    gt, _, _ = ob.sql_topk(x, q, 10)
    rec = np.mean([len(set(rows[i].tolist()) & set(gt[i].tolist())) / 10 for i in range(len(q))])
    assert rec >= 0.95


def test_merge_topk_host_orders_by_distance_then_row():
    rows = np.array([[[5, 9, 0]], [[7, 2, 0]]], np.uint64)      # 2 shards, 1 query, k=3
    dist = np.array([[[0.1, 0.5, 0.0]], [[0.1, 0.2, 0.0]]], np.float32)
    cnt = np.array([[2], [2]], np.uint32)
    r, d, c = merge_topk_host(rows, dist, cnt, 3)
    assert r[0].tolist() == [5, 7, 2] and c[0] == 3
    # lists are consumed in their given order: a tie inside one shard is not re-sorted by row id
    rows = np.array([[[9, 5]], [[7, 7]]], np.uint64)
    dist = np.array([[[1.0, 1.0]], [[1.0, 2.0]]], np.float32)
    r, d, c = merge_topk_host(rows, dist, np.array([[2], [2]], np.uint32), 3)
    assert r[0].tolist() == [7, 9, 5]
    assert shard_bounds(10, 3, 0) == (0, 3) and shard_bounds(10, 3, 2) == (6, 10)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _sharded_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    n_total, dim, nq, k, ef = 2000, 16, 32, 5, 32
    x = ds.gaussian_latent(n_total, dim, seed=21)
    q = ds.gaussian_latent(nq, dim, seed=22)
    lo, hi = shard_bounds(n_total, world, rank)
    g = ob.OracleGraph.build(x[lo:hi], seed=30 + rank, row_ids=np.arange(lo, hi, dtype=np.uint64))

    def local_search(queries, o_rows, o_dd, o_cnt):  # the rank's top-k goes straight into its packed block
        rows, _, dd, cnt, _ = g.search(queries, k, ef)
        o_rows.copy_(torch.from_numpy(rows.astype(np.int64)))
        o_dd.copy_(torch.from_numpy(dd.copy()))
        o_cnt.copy_(torch.from_numpy(cnt.astype(np.int32)))

    def merge(gathered, block_bytes):  # ONE all-gather delivered [world, block]; the host specification merges it
        assert gathered.numel() == world * block_bytes
        g_rows, g_dd, g_cnt = s.unpack(gathered)
        r, d, c = merge_topk_host(g_rows.numpy().astype(np.uint64), g_dd.numpy(), g_cnt.numpy().astype(np.uint32), k)
        return torch.from_numpy(r.astype(np.int64)), torch.from_numpy(d), torch.from_numpy(c.astype(np.int32))

    s = ShardedSearch(dist, world, local_search, merge, nq, k, "cpu")
    rows, dd, cnt = s.search_batch(q)
    np.savez(os.path.join(out_dir, f"rank{rank}.npz"), rows=rows.numpy(), dist=dd.numpy(), cnt=cnt.numpy())
    dist.destroy_process_group()


def test_sharded_search_world2_gloo(tmp_path):
    world = 2
    port = _free_port()
    mp.spawn(_sharded_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    r0 = np.load(tmp_path / "rank0.npz")
    r1 = np.load(tmp_path / "rank1.npz")
    assert np.array_equal(r0["rows"], r1["rows"]) and np.array_equal(r0["dist"], r1["dist"])
    # the merged answer equals merging the per-shard oracle results in one process
    n_total, dim, nq, k, ef = 2000, 16, 32, 5, 32
    x = ds.gaussian_latent(n_total, dim, seed=21)
    q = ds.gaussian_latent(nq, dim, seed=22)
    parts = []
    for rank in range(world):
        lo, hi = shard_bounds(n_total, world, rank)
        g = ob.OracleGraph.build(x[lo:hi], seed=30 + rank, row_ids=np.arange(lo, hi, dtype=np.uint64))
        parts.append(g.search(q, k, ef))
    rows = np.stack([p[0] for p in parts])
    dd = np.stack([p[2] for p in parts])
    cnt = np.stack([p[3] for p in parts])
    mr, md, mc = merge_topk_host(rows, dd, cnt, k)
    assert np.array_equal(mr.astype(np.int64), r0["rows"]) and np.array_equal(md, r0["dist"])
    # and it is close to the exact global answer
    gt, _, _ = ob.sql_topk(x, q, k)
    rec = np.mean([len(set(r0["rows"][i].tolist()) & set(gt[i].astype(np.int64).tolist())) / k for i in range(nq)])
    assert rec >= 0.9


def test_partitioned_builder_keeps_structure():
    """graph_build's IVF candidate pass (large corpora): same structural contract as the all-pairs pass."""
    import torch
    from turdb_b200 import datasets as ds
    from turdb_b200.graph_build import build_graph
    torch.set_num_threads(4)
    x = ds.gaussian_latent(6000, 32, seed=3)
    a = build_graph(x, seed=5, device="cpu", ivf_cells=32, ivf_probe=6, ivf_exact_prefix=512)
    assert a["provenance"].endswith("(ivf 32x6)")
    n = 6000
    assert a["l0_adj"].shape == (n, 32) and a["l0_cnt"].max() <= 32 and a["l0_cnt"].min() >= 1
    valid = np.arange(32)[None, :] < a["l0_cnt"][:, None]
    assert (a["l0_adj"][valid] < n).all() and (a["l0_adj"][~valid] == 0xFFFFFFFF).all()
    assert not (a["l0_adj"] == np.arange(n, dtype=np.uint32)[:, None]).any()  # no self loops
    assert a["levels"][a["entry"]] == a["max_level"]


def test_bench_rank0_only_section_issues_no_collectives():
    """bench.py keeps rank 0's GPU busy a little longer for the clock sampler; that rank-0-only section once called
    the sharded step (all-gather) and deadlocked every N>1 run.  It may only launch rank-local work."""
    import os
    src = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bench.py")).read()
    block = src[src.index("keep the GPU under the same load"):src.index("clocks = sampler.stop()")]
    assert "local_search(" in block
    for forbidden in ("step(", "sharded.", "dist.", "barrier("):
        assert forbidden not in block, forbidden


def test_bench_dump_outputs_are_float_and_a_seeded_sample_when_large(tmp_path, monkeypatch):
    import bench
    rows = np.arange(40, dtype=np.int64).reshape(20, 2)
    rows[3, 1] = -1
    arrays = {"rows": rows, "distances": np.linspace(0, 1, 40, dtype=np.float32).reshape(20, 2),
              "counts": np.full(20, 2, np.int32)}
    bench.dump_outputs(str(tmp_path / "all"), arrays, seed=1)
    got = {k: np.load(tmp_path / "all" / f"{k}.npy") for k in ("query_index", "rows", "distances", "counts")}
    assert got["distances"].dtype == np.float32 and got["rows"].dtype == got["counts"].dtype == np.float64
    assert np.array_equal(got["rows"], rows) and np.array_equal(got["query_index"], np.arange(20))
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 200)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays, seed=1)
    qa, qb = (np.load(tmp_path / d / "query_index.npy") for d in ("a", "b"))
    assert np.array_equal(qa, qb) and 0 < len(qa) < 20
    assert sum(np.load(f).nbytes for f in (tmp_path / "a").iterdir()) <= 200
    assert np.array_equal(np.load(tmp_path / "a" / "rows.npy"), rows[qa.astype(np.int64)])
