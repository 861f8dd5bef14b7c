"""The SQL distance-range scan (turdb_cuda_sql_range_batch) at serving size, against the top-k statement on the same data.

Corpus: config 2 of bench.py (1M x 384 latent-Gaussian, L2-normalised), `<=>` (cosine).  10k statements
`WHERE emb <=> literal < r_q LIMIT 10`; per radius class, r_q is the value of the statement's t-th nearest row (f64
cosine distance from numpy on a sample of the corpus, scaled up to the full size), so that about t = 10, 100 and 1000
rows qualify.  For each class, range batches and `ORDER BY emb <=> literal LIMIT 10` batches (turdb_cuda_sql_topk_batch,
the same literals) are alternated; every call is timed on the host clock and ends in a device synchronise.  Reported:
ms per batch (median, min), the mean count of qualifying rows, how many statements took the streaming fallback
(TURDB_EXACT_VERBOSE line of one extra call), and the filter kernel's device time (torch.profiler, separate calls) as
TFLOP/s (2 nq n kp / time) against the 2,250 TFLOP/s BF16/FP16 dense data-sheet figure of one B200.

    python tools/range_probe.py --out /tmp/range_probe.json
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

BF16_PEAK_TFLOPS = 2250.0


def card() -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [f.strip() for f in out.split(",")]
        return {"name": name, "power_limit": power, "sm_clock_max": clock}
    except Exception as e:  # the record still says where it came from
        return {"name": None, "error": str(e)}


def fallback_count(fn) -> dict:
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
    m = re.search(r"\[turdb range\] statements=(\d+) fallback=(\d+) cap=(\d+)", text)
    form = re.search(r"form=(\S+) tile_n=(\d+)", text)
    return {"fallback": int(m.group(2)) if m else None, "capacity": int(m.group(3)) if m else None,
            "filter_form": form.group(1) if form else None}


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
    from turdb_b200.sql_operator import RangeCmp, VectorOp, VectorRangeScanBatch, VectorScanBatch

    if not torch.cuda.is_available():
        sys.exit("range_probe needs a CUDA device")
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

    rng_op = VectorRangeScanBatch(idx, VectorOp.CosineDistance, RangeCmp.Lt, 10)
    topk_op = VectorScanBatch(idx, VectorOp.CosineDistance, 10)
    kp = (dim + 63) // 64 * 64

    def timed(fn):
        torch.cuda.synchronize()
        t = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t) * 1e3, out

    rec = {"tool": "range_probe", "card": card(), "corpus": f"{n}x{dim} gaussian_latent(seed=1, normalised), cosine",
           "statements": nq, "limit": 10, "bf16_peak_tflops_datasheet": BF16_PEAK_TFLOPS, "classes": []}
    topk_op.execute(q)  # warm-up: module load, the 16-bit cosine copy
    for t, r in radii.items():
        rng_op.execute(q, r)
        ms_range, ms_topk, counts = [], [], None
        for _ in range(args.reps):
            dt, (_, _, counts) = timed(lambda: rng_op.execute(q, r))
            ms_range.append(dt)
            dt, _ = timed(lambda: topk_op.execute(q))
            ms_topk.append(dt)
        fb = fallback_count(lambda: rng_op.execute(q, r))
        # device time of the filter pass (and of every other kernel of the call), separate calls under the profiler
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                rng_op.execute(q, r)
            torch.cuda.synchronize()
        kern = {}
        for ev in prof.key_averages():
            if ev.device_type.name == "CUDA" and ev.count:
                kern[ev.key[:80]] = round(getattr(ev, "device_time_total", getattr(ev, "cuda_time_total", 0.0)) / 1e3 / 3, 4)
        filt_ms = sum(v for k, v in kern.items() if "exact_gemm_filter" in k)
        tflops = 2.0 * nq * n * kp / (filt_ms * 1e-3) / 1e12 if filt_ms else None
        c = {"target_rows": t, "mean_qualifying": float(np.mean(counts)), "median_qualifying": float(np.median(counts)),
             "max_qualifying": int(np.max(counts)),
             "range_ms_median": float(np.median(ms_range)), "range_ms_min": float(np.min(ms_range)),
             "topk_limit10_ms_median": float(np.median(ms_topk)), "topk_limit10_ms_min": float(np.min(ms_topk)),
             **fb, "kernel_ms_per_call": kern, "filter_ms": filt_ms,
             "filter_tflops": tflops, "filter_share_of_bf16_peak": tflops / BF16_PEAK_TFLOPS if tflops else None}
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
