"""The nearest rows within a radius (turdb_cuda_sql_range_topk_batch) at serving size, against the range scan and the
top-k statement on the same batch.

Corpus: config 2 of bench.py (1M x 384 latent-Gaussian, L2-normalised), `<=>` (cosine).  10k statements
`WHERE emb <=> literal < r_q ORDER BY emb <=> literal LIMIT 10`; per radius class, r_q is the value of the statement's
t-th nearest row (f64 cosine distance on a sample of the corpus, scaled up to the full size), so that about t = 10, 100
and 1000 rows qualify.  For each class, three calls on the same literals are alternated: the range top-k, the range scan
`WHERE emb <=> literal < r_q LIMIT 10` (turdb_cuda_sql_range_batch) and `ORDER BY emb <=> literal LIMIT 10`
(turdb_cuda_sql_topk_batch).  Every call is timed on the host clock and ends in a device synchronise.  Reported: ms per
batch (median, min), the mean count of qualifying rows, how many statements took the streaming fallback
(TURDB_EXACT_VERBOSE line of one extra call of each range kind), and every kernel's device time per range top-k call
(torch.profiler, separate calls).  The card's name and power limit are read in the same run.

    python tools/range_topk_probe.py --out /tmp/range_topk_probe.json
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

from range_probe import card, fallback_count  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--dim", type=int, default=384)
    ap.add_argument("--nq", type=int, default=10_000)
    ap.add_argument("--targets", default="10,100,1000", help="rows that should qualify per statement")
    ap.add_argument("--reps", type=int, default=5, help="timed calls of each kind per class (alternated)")
    ap.add_argument("--sample", type=int, default=100_000, help="corpus rows used to choose the radii")
    ap.add_argument("--out", default="")
    args = ap.parse_args()

    import torch
    from turdb_b200 import datasets as ds
    from turdb_b200.hnsw import CudaHnswIndex
    from turdb_b200.sql_operator import RangeCmp, VectorOp, VectorRangeScanBatch, VectorRangeTopKBatch, VectorScanBatch

    if not torch.cuda.is_available():
        sys.exit("range_topk_probe needs a CUDA device")
    n, dim, nq = args.n, args.dim, args.nq
    x = ds.gaussian_latent(n, dim, seed=1, normalise=True)
    q = ds.gaussian_latent(nq, dim, seed=2, normalise=True)
    g = dict(vectors=x, row_ids=np.arange(n, dtype=np.uint64), levels=np.zeros(n, np.uint8),
             l0_adj=np.full((n, 32), 0xFFFFFFFF, np.uint32), l0_cnt=np.zeros(n, np.uint8),
             up_base=np.full(n, 0xFFFFFFFF, np.uint32), up_adj=np.zeros((0, 16), np.uint32), up_cnt=np.zeros(0, np.uint8),
             entry=0, max_level=0)
    idx = CudaHnswIndex.from_graph(g)

    # radii: the t-th smallest cosine distance over the full corpus ~ the (t * sample / n)-th over a sample
    xs = torch.from_numpy(x[:: max(1, n // args.sample)]).cuda().double()
    qd = torch.from_numpy(q).cuda().double()
    scale = xs.shape[0] / n
    radii = {}
    for t in [int(v) for v in args.targets.split(",")]:
        kk = max(1, int(round(t * scale)))
        r = torch.empty(nq, dtype=torch.float64)
        for b in range(0, nq, 1000):
            d = 1.0 - qd[b:b + 1000] @ xs.T
            r[b:b + 1000] = torch.kthvalue(d, kk, dim=1).values.cpu()
        radii[t] = r.numpy()
    del xs, qd

    cos = VectorOp.CosineDistance
    rtk_op = VectorRangeTopKBatch(idx, cos, RangeCmp.Lt, cos, 10)
    rng_op = VectorRangeScanBatch(idx, cos, RangeCmp.Lt, 10)
    topk_op = VectorScanBatch(idx, cos, 10)

    def timed(fn):
        torch.cuda.synchronize()
        t = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t) * 1e3, out

    rec = {"tool": "range_topk_probe", "card": card(), "corpus": f"{n}x{dim} gaussian_latent(seed=1, normalised), cosine",
           "statements": nq, "limit": 10, "classes": []}
    topk_op.execute(q)  # warm-up: module load, the 16-bit cosine copy
    for t, r in radii.items():
        rtk_op.execute(q, r)
        rng_op.execute(q, r)
        ms_rtk, ms_range, ms_topk, counts, returned = [], [], [], None, None
        for _ in range(args.reps):
            dt, (_, _, returned) = timed(lambda: rtk_op.execute(q, r))
            ms_rtk.append(dt)
            dt, (_, _, counts) = timed(lambda: rng_op.execute(q, r))
            ms_range.append(dt)
            dt, _ = timed(lambda: topk_op.execute(q))
            ms_topk.append(dt)
        fb_rtk = fallback_count(lambda: rtk_op.execute(q, r))
        fb_rng = fallback_count(lambda: rng_op.execute(q, r))
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                rtk_op.execute(q, r)
            torch.cuda.synchronize()
        kern = {}
        for ev in prof.key_averages():
            if ev.device_type.name == "CUDA" and ev.count:
                kern[ev.key[:80]] = round(getattr(ev, "device_time_total", getattr(ev, "cuda_time_total", 0.0)) / 1e3 / 3, 4)
        c = {"target_rows": t, "mean_qualifying": float(np.mean(counts)), "median_qualifying": float(np.median(counts)),
             "max_qualifying": int(np.max(counts)), "mean_returned": float(np.mean(returned)),
             "range_topk_ms_median": float(np.median(ms_rtk)), "range_topk_ms_min": float(np.min(ms_rtk)),
             "range_ms_median": float(np.median(ms_range)), "range_ms_min": float(np.min(ms_range)),
             "topk_limit10_ms_median": float(np.median(ms_topk)), "topk_limit10_ms_min": float(np.min(ms_topk)),
             "range_topk_fallback": fb_rtk["fallback"], "range_fallback": fb_rng["fallback"],
             "capacity": fb_rtk["capacity"], "filter_form": fb_rtk["filter_form"],
             "range_topk_kernel_ms_per_call": kern,
             "range_topk_filter_ms": sum(v for k, v in kern.items() if "exact_gemm_filter" in k),
             "range_topk_kernel_ms": sum(v for k, v in kern.items() if "sql_range_topk_kernel" in k)}
        rec["classes"].append(c)
        print(json.dumps(c), flush=True)
    idx.close()
    print(json.dumps(rec))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
