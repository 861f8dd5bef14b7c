"""Compacting a resident index (turdb_cuda_index_compact): what a compaction costs against rebuilding the live rows
(turdb_cuda_index_build), and what it gives back to the traversal after 1 % and 10 % of the rows were deleted.

Corpus and graph: config 2 of bench.py (1M x 384 latent-Gaussian, L2-normalised, cosine; graph by the device insert
path, M 16, efC 100, steps of <= 4096 nodes), built once and uploaded per measurement (turdb_cuda_index_create).  Per
deletion level (a seeded random choice of rows):
  - compaction time: host clock around the call, which ends in a device synchronise; median over fresh uploads;
  - rebuild time: turdb_cuda_index_build over the live rows (same parameters), host clock, in the same run;
  - the bench-shaped traversal (10k queries, ef 128, k 10, device entry) before compaction (search_filtered over live),
    after it, and on the index without deletions, alternated; recall@10 against the exact top-10 of the live rows for
    the filtered search, the compacted graph and the rebuilt graph;
  - `ORDER BY emb <=> literal LIMIT 10` and the range scan `WHERE emb <=> literal < r LIMIT 10` (r about the 10th nearest
    row's distance) over 10k statements, before and after compaction.

    python tools/compact_probe.py --out /tmp/compact_probe.json
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from delete_probe import card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--dim", type=int, default=384)
    ap.add_argument("--nq", type=int, default=10_000)
    ap.add_argument("--ef", type=int, default=128)
    ap.add_argument("--reps", type=int, default=5, help="timed calls of each traversal / statement kind (alternated)")
    ap.add_argument("--compact-reps", type=int, default=3, help="fresh uploads compacted per deletion level")
    ap.add_argument("--seed", type=int, default=20261018)
    ap.add_argument("--out", default="")
    args = ap.parse_args()

    import torch
    from turdb_b200 import datasets as ds
    from turdb_b200.hnsw import CudaHnswIndex, DistanceFunction
    from turdb_b200.sql_operator import RangeCmp, VectorOp, VectorRangeScanBatch, VectorScanBatch

    if not torch.cuda.is_available():
        sys.exit("compact_probe needs a CUDA device")
    n, dim, nq, k = args.n, args.dim, args.nq, 10
    cos = DistanceFunction.Cosine
    rec = {"tool": "compact_probe", "card": card(),
           "corpus": f"{n}x{dim} gaussian_latent(seed={args.seed + 1000}, normalised), cosine",
           "graph": "device insert path, M 16, efC 100, mode 1, steps of <= 4096 nodes", "statements": nq, "ef": args.ef,
           "k": k, "reps": args.reps, "compact_reps": args.compact_reps}
    x = ds.gaussian_latent(n, dim, seed=args.seed + 1000, normalise=True)
    q = ds.gaussian_latent(nq, dim, seed=args.seed + 7, normalise=True)
    rid = np.arange(n, dtype=np.uint64)
    rnd = 1.0 - np.random.default_rng(args.seed).random(n)
    built = CudaHnswIndex.build(x, rid, rnd, m=16, ef_construction=100, mode=1, max_batch=4096, metric=cos)
    arrays = built.export_graph()
    built.close()

    def sync_ms(fn):
        torch.cuda.synchronize()
        t = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t) * 1e3, out

    xd = torch.from_numpy(x).cuda()
    radii = np.empty(nq)
    for b in range(0, nq, 1000):
        sim = torch.from_numpy(q[b:b + 1000]).cuda() @ xd.T
        radii[b:b + 1000] = (1.0 - torch.topk(sim, 10, dim=1).values[:, -1].double()).cpu().numpy()
    del xd, sim

    dq = torch.from_numpy(q).cuda()
    d_rows = torch.empty((nq, k), dtype=torch.int64, device="cuda")
    d_dist = torch.empty((nq, k), dtype=torch.float32, device="cuda")
    d_cnt = torch.empty(nq, dtype=torch.int32, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream

    def traversal(ix):
        ix.search_batch_device(dq.data_ptr(), nq, k, args.ef, cos, d_rows.data_ptr(), d_dist.data_ptr(), d_cnt.data_ptr(),
                               stream=stream)
        return d_rows

    def recall(ix, truth):
        traversal(ix)
        torch.cuda.synchronize()
        got = d_rows.cpu().numpy().view(np.uint64)
        return float(np.mean([len(set(got[i].tolist()) & set(truth[i].tolist())) / k for i in range(nq)]))

    def timed(work, ix, base):
        """median ms of each statement kind on ix, alternated with base (warmed first)"""
        out = {}
        for name, fn in work.items():
            fn(base)
            fn(ix)
            mine, other = [], []
            for _ in range(args.reps):
                other.append(sync_ms(lambda: fn(base))[0])
                mine.append(sync_ms(lambda: fn(ix))[0])
            out[name] = (float(np.median(mine)), float(np.median(other)))
        return out

    work = {"search": traversal,
            "sql_topk_limit10": lambda i: VectorScanBatch(i, VectorOp.CosineDistance, k).execute(q),
            "range_about10": lambda i: VectorRangeScanBatch(i, VectorOp.CosineDistance, RangeCmp.Lt, k).execute(q, radii)}
    base = CudaHnswIndex.from_graph(arrays, metric=cos)
    rec["levels"] = []
    for frac in (0.01, 0.10):
        dead = np.random.default_rng(args.seed + int(frac * 1000)).random(n) < frac
        live = np.flatnonzero(~dead)
        lvl = {"deleted_fraction": frac, "deleted_rows": int(dead.sum())}
        # compaction on fresh uploads
        ts = []
        for _ in range(args.compact_reps):
            ix = CudaHnswIndex.from_graph(arrays, metric=cos)
            ix.delete(np.flatnonzero(dead))
            bytes_before = ix.info()["device_bytes"]
            ms, o2n = sync_ms(ix.compact)
            ts.append(ms)
            bytes_after = ix.info()["device_bytes"]
            ix.close()
        lvl["compact_ms_median"] = float(np.median(ts))
        lvl["compact_ms_all"] = ts
        lvl["device_bytes_before_after"] = [bytes_before, bytes_after]
        rb_ms, rebuilt = sync_ms(lambda: CudaHnswIndex.build(x[live], rid[live], rnd[live], m=16, ef_construction=100,
                                                              mode=1, max_batch=4096, metric=cos))
        lvl["rebuild_live_rows_ms"] = rb_ms
        print(json.dumps(lvl), flush=True)

        # before (filtered) / after compaction, each alternated with the index without deletions
        filt = CudaHnswIndex.from_graph(arrays, metric=cos)
        filt.delete(np.flatnonzero(dead))
        truth = filt.bruteforce_topk(q, k, cos)[0]  # the exact top-10 of the live rows (row ids)
        lvl["recall_at_10_filtered"] = recall(filt, truth)
        before = timed(work, filt, base)
        comp = CudaHnswIndex.from_graph(arrays, metric=cos)
        comp.delete(np.flatnonzero(dead))
        comp.compact()
        lvl["recall_at_10_compacted"] = recall(comp, truth)
        lvl["recall_at_10_rebuilt"] = recall(rebuilt, truth)
        after = timed(work, comp, base)
        for name in work:
            lvl[f"{name}_ms_before_compaction"] = before[name][0]
            lvl[f"{name}_ms_after_compaction"] = after[name][0]
            lvl[f"{name}_ms_no_deletions_same_run"] = float(np.median([before[name][1], after[name][1]]))
        lvl["search_ms_no_deletions_scaled_by_live_share"] = lvl["search_ms_no_deletions_same_run"] * len(live) / n
        rec["levels"].append(lvl)
        print(json.dumps(lvl), flush=True)
        for ix in (filt, comp, rebuilt):
            ix.close()
    base.close()
    print(json.dumps(rec))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
