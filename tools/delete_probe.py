"""Deleting rows from a resident index (turdb_cuda_index_delete): what a delete call costs, and what 1 % and 10 % of
deleted rows cost every read path, against the same index without deletions.

Corpus and graph: config 2 of bench.py (1M x 384 latent-Gaussian, L2-normalised, cosine; graph by the device insert
path, M 16, efC 100, steps of <= 4096 nodes).  The graph is built once and uploaded three times (turdb_cuda_index_create):
0 %, 1 % and 10 % of the rows deleted (a seeded random choice).  Measured:
  - delete latency for calls of 1, 1000 and 100k ids on a fourth upload (the first call allocates the bitmap);
  - per deletion level, alternated with the 0 % index in the same run: the bench-shaped traversal (10k queries, ef 128,
    k 10, device entry) with recall@10 against the exact top-10 of the live rows (the certified exact path on the same
    index), `ORDER BY emb <=> literal LIMIT 10` over 10k statements (exact scan) and the range scan
    `WHERE emb <=> literal < r LIMIT 10` with r about the 10th nearest row's distance;
  - how many statements the streaming scan redid (TURDB_EXACT_VERBOSE lines of one extra call each).
Every time is the median of host-clock times of calls that end in a device synchronise.

    python tools/delete_probe.py --out /tmp/delete_probe.json
"""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card() -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [f.strip() for f in out.split(",")]
        return {"name": name, "power_limit": power, "sm_clock_max": clock}
    except Exception as e:  # the record still says where it came from
        return {"name": None, "error": str(e)}


def fallback_count(fn, what: str):
    """One call with TURDB_EXACT_VERBOSE set, its stderr captured at the file-descriptor level."""
    os.environ["TURDB_EXACT_VERBOSE"] = "1"
    with tempfile.TemporaryFile() as f:
        saved = os.dup(2)
        os.dup2(f.fileno(), 2)
        try:
            fn()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["TURDB_EXACT_VERBOSE"]
        f.seek(0)
        text = f.read().decode(errors="replace")
    m = re.search(rf"\[turdb {what}\] statements=(\d+) fallback=(\d+)", text)
    return int(m.group(2)) if m else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--dim", type=int, default=384)
    ap.add_argument("--nq", type=int, default=10_000)
    ap.add_argument("--ef", type=int, default=128)
    ap.add_argument("--reps", type=int, default=5, help="timed calls of each kind and index (alternated)")
    ap.add_argument("--seed", type=int, default=20261018)
    ap.add_argument("--out", default="")
    args = ap.parse_args()

    import torch
    from turdb_b200 import datasets as ds
    from turdb_b200.hnsw import CudaHnswIndex, DistanceFunction
    from turdb_b200.sql_operator import RangeCmp, VectorOp, VectorRangeScanBatch, VectorScanBatch

    if not torch.cuda.is_available():
        sys.exit("delete_probe needs a CUDA device")
    n, dim, nq, k = args.n, args.dim, args.nq, 10
    cos = DistanceFunction.Cosine
    rec = {"tool": "delete_probe", "card": card(), "corpus": f"{n}x{dim} gaussian_latent(seed={args.seed + 1000}, normalised), cosine",
           "graph": "device insert path, M 16, efC 100, mode 1, steps of <= 4096 nodes", "statements": nq, "ef": args.ef,
           "k": k, "reps": args.reps}
    x = ds.gaussian_latent(n, dim, seed=args.seed + 1000, normalise=True)
    q = ds.gaussian_latent(nq, dim, seed=args.seed + 7, normalise=True)
    rid = np.arange(n, dtype=np.uint64)
    built = CudaHnswIndex.build(x, rid, None, m=16, ef_construction=100, mode=1, max_batch=4096, metric=cos, seed=args.seed)
    arrays = built.export_graph()
    built.close()

    def sync_ms(fn):
        torch.cuda.synchronize()
        t = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t) * 1e3, out

    # delete latency
    rng = np.random.default_rng(args.seed)
    lat = CudaHnswIndex.from_graph(arrays, metric=cos)
    first = rng.choice(n, 1)
    first_ms, _ = sync_ms(lambda: lat.delete(first))
    rec["delete_ms"] = {"first_call_1_row_allocates": first_ms}
    for size in (1, 1000, 100_000):
        batches = [rng.choice(n, size, replace=False) for _ in range(args.reps)]  # drawn outside the timed region
        ts = [sync_ms(lambda: lat.delete(ids))[0] for ids in batches]
        rec["delete_ms"][f"{size}_rows_median"] = float(np.median(ts))
        rec["delete_ms"][f"{size}_rows_min"] = float(np.min(ts))
    rec["delete_ms"]["deleted_after"] = lat.delete([])
    lat.close()
    print(json.dumps(rec["delete_ms"]), flush=True)

    # range radii: about the 10th nearest row's cosine distance (f32 matmul on the device; approximate on purpose)
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

    base = CudaHnswIndex.from_graph(arrays, metric=cos)
    rec["levels"] = []
    for frac in (0.0, 0.01, 0.10):
        ix = CudaHnswIndex.from_graph(arrays, metric=cos)
        dead = np.random.default_rng(args.seed + int(frac * 1000)).random(n) < frac
        if frac:
            assert ix.delete(np.flatnonzero(dead)) == int(dead.sum())
        work = {"search": traversal,
                "sql_topk_limit10": lambda i: VectorScanBatch(i, VectorOp.CosineDistance, k).execute(q),
                "range_about10": lambda i: VectorRangeScanBatch(i, VectorOp.CosineDistance, RangeCmp.Lt, k).execute(q, radii)}
        lvl = {"deleted_fraction": frac, "deleted_rows": int(dead.sum())}
        for name, fn in work.items():
            fn(base)
            fn(ix)  # warm-up: modules, 16-bit copies, visited-set sizing
            mine, zero = [], []
            for _ in range(args.reps):
                zero.append(sync_ms(lambda: fn(base))[0])
                mine.append(sync_ms(lambda: fn(ix))[0])
            lvl[f"{name}_ms_median"] = float(np.median(mine))
            lvl[f"{name}_ms_median_0pct_same_run"] = float(np.median(zero))
        gt = ix.bruteforce_topk(q, k, cos)[0]  # the exact top-10 of the live rows
        traversal(ix)
        torch.cuda.synchronize()
        got = d_rows.cpu().numpy().view(np.uint64)
        lvl["recall_at_10"] = float(np.mean([len(set(got[i].tolist()) & set(gt[i].tolist())) / k for i in range(nq)]))
        lvl["returned_deleted_rows"] = int(dead[got[got < n].astype(np.int64)].sum())
        lvl["sql_topk_fallback"] = fallback_count(lambda: work["sql_topk_limit10"](ix), "topk")
        lvl["range_fallback"] = fallback_count(lambda: work["range_about10"](ix), "range")
        lvl["range_mean_count"] = float(np.mean(work["range_about10"](ix)[2]))
        rec["levels"].append(lvl)
        print(json.dumps(lvl), flush=True)
        ix.close()
    base.close()
    print(json.dumps(rec))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
