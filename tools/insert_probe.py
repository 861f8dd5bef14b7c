"""Appending rows to a resident index (turdb_cuda_index_insert): throughput per call size, and the search quality of the
grown graph against one build over the same rows.

Corpus: config 2 of bench.py (1M x 384 latent-Gaussian, L2-normalised, cosine).  The first n - tail rows are built with
turdb_cuda_index_build (steps of <= --build-batch nodes); the tail is appended in calls of 1, 64, 4096 and 100k rows
(--calls sets how many calls of each size).  Each call is timed on the host clock and ends in a device synchronise.
Then one build over all n rows with the same parameters, and both indexes searched with the same queries at ef 128:
recall@10 against the exact top-10 (the certified exact path) and the traversal's kernel time (per-launch device events).

    python tools/insert_probe.py --out /tmp/insert_probe.json
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--dim", type=int, default=384)
    ap.add_argument("--latent", type=int, default=16)
    ap.add_argument("--seed", type=int, default=20261018)
    ap.add_argument("--m", type=int, default=16)
    ap.add_argument("--ef-construction", type=int, default=100)
    ap.add_argument("--build-batch", type=int, default=4096)
    ap.add_argument("--sizes", default="1,64,4096,100000", help="rows per insert call")
    ap.add_argument("--calls", default="200,50,5,1", help="calls of each size")
    ap.add_argument("--nq", type=int, default=10_000)
    ap.add_argument("--ef", type=int, default=128)
    ap.add_argument("--out", default="")
    args = ap.parse_args()

    import torch
    from turdb_b200 import datasets as ds
    from turdb_b200.hnsw import CudaHnswIndex, DistanceFunction

    if not torch.cuda.is_available():
        sys.exit("insert_probe needs a CUDA device")
    sizes = [int(s) for s in args.sizes.split(",")]
    calls = [int(c) for c in args.calls.split(",")]
    tail = sum(s * c for s, c in zip(sizes, calls))
    n, k0 = args.n, args.n - tail
    if k0 < 1:
        sys.exit(f"the tail ({tail} rows) does not fit n = {n}")
    x = ds.gaussian_latent(n, args.dim, seed=args.seed + 1000, latent=args.latent, normalise=True)
    q = ds.gaussian_latent(args.nq, args.dim, seed=args.seed + 7, latent=args.latent, normalise=True)
    rid = np.arange(n, dtype=np.uint64)
    rnd = 1.0 - np.random.default_rng(args.seed).random(n)
    params = dict(m=args.m, ef_construction=args.ef_construction, mode=1, max_batch=args.build_batch)
    cos = DistanceFunction.Cosine

    def sync_time(fn):
        torch.cuda.synchronize()
        t = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        return time.perf_counter() - t

    rec = {"tool": "insert_probe", "card": card(), "corpus": f"{n}x{args.dim} gaussian_latent(latent={args.latent}, normalised)",
           "seed": args.seed, "params": params, "prefix_rows": k0, "tail_rows": tail}
    t = time.perf_counter()
    idx = CudaHnswIndex.build(x[:k0], rid[:k0], rnd[:k0], metric=cos, **params)
    torch.cuda.synchronize()
    rec["prefix_build_s"] = time.perf_counter() - t
    s = k0
    per_size = []
    for size, count in zip(sizes, calls):
        times, grew = [], 0
        for _ in range(count):
            before = idx.info()["device_bytes"]
            times.append(sync_time(lambda: idx.insert(x[s:s + size], rid[s:s + size], rnd[s:s + size], max_batch=args.build_batch)))
            grew += idx.info()["device_bytes"] != before
            s += size
        t = np.array(times)
        per_size.append({"rows_per_call": size, "calls": count, "median_ms": float(np.median(t) * 1e3),
                         "min_ms": float(t.min() * 1e3), "max_ms": float(t.max() * 1e3),
                         "rows_per_s": float(size / np.median(t)), "calls_that_grew": grew})
        print(json.dumps(per_size[-1]), flush=True)
    assert s == n and idx.info()["n"] == n
    rec["insert"] = per_size
    rec["device_bytes_appended"] = idx.info()["device_bytes"]

    t = time.perf_counter()
    full = CudaHnswIndex.build(x, rid, rnd, metric=cos, **params)
    torch.cuda.synchronize()
    rec["full_build_s"] = time.perf_counter() - t
    rec["device_bytes_full"] = full.info()["device_bytes"]

    gt_rows = full.bruteforce_topk(q, 10, cos)[0]

    def quality(index):
        index.search_batch(q, 10, args.ef, cos)  # warm-up: module load, visited-table sizing
        index.profile_begin(8)
        for _ in range(3):
            rows = index.search_batch(q, 10, args.ef, cos, want_stats=False)[0]
        torch.cuda.synchronize()
        main_ms, ovf_ms = index.profile_read(8)
        recall = float(np.mean([len(set(rows[i].tolist()) & set(gt_rows[i].tolist())) / 10 for i in range(len(q))]))
        return {"recall_at_10": recall, "kernel_ms_median": float(np.median(main_ms + ovf_ms))}
    rec["search_ef"] = args.ef
    rec["nq"] = args.nq
    rec["appended"] = quality(idx)
    rec["full_build"] = quality(full)
    print(json.dumps(rec))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
