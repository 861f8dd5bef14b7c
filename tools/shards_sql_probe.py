"""Exact `ORDER BY emb <-> literal LIMIT 10` over a table split into sub-indexes (turdb_cuda_shards_sql_topk_batch)
against the same statements on ONE index of the same rows (turdb_cuda_sql_topk_batch, exact scan).

Corpus: config 5's shape, 128-d L2 clustered rows (1000 centres per 100k rows), `--rows` per shard; `--shards` lists
the shard counts to run, all shards on device 0 (or spread over `--devices` GPUs).  10k statements per batch, literals
near corpus rows.  For each shard count the sharded and the single-index calls are alternated, `--reps` each; every call
is timed on the host clock and ends in a device synchronise (H2D of the literals and D2H of the results included).
Both results are compared bit for bit.  One profiled call of the sharded form (torch.profiler, separate) gives every
kernel's device time summed over shards, and two spans: from the first kernel to the last one that ended before the
first relay kernel began, and from that relay kernel to the end of the emit kernel.  With several shards on one device
the filters and relays overlap, so there the kernel sums are the split to read.  One TURDB_EXACT_VERBOSE call gives each
shard's fallback count.  The card's name and power limit are read in the same run.

    python tools/shards_sql_probe.py --rows 12500000 --shards 2,4 --out /tmp/shards_sql_probe.json
"""
from __future__ import annotations

import argparse
import json
import os
import re
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from range_probe import card  # noqa: E402


def verbose_fallbacks(fn) -> list[int]:
    """One call with TURDB_EXACT_VERBOSE set, stderr captured at the file-descriptor level -> fallback count per shard."""
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
    return [int(m.group(1)) for m in re.finditer(r"\[turdb shards_topk shard \d+\] statements=\d+ fallback=(\d+)", text)]


def table_index(x, row_ids, device=0):
    from turdb_b200.hnsw import CudaHnswIndex
    n = x.shape[0]
    g = dict(vectors=x, row_ids=row_ids, levels=np.zeros(n, np.uint8), l0_adj=np.full((n, 32), 0xFFFFFFFF, np.uint32),
             l0_cnt=np.zeros(n, np.uint8), up_base=np.full(n, 0xFFFFFFFF, np.uint32), up_adj=np.zeros((0, 16), np.uint32),
             up_cnt=np.zeros(0, np.uint8), entry=0, max_level=0)
    return CudaHnswIndex.from_graph(g, device=device)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=12_500_000, help="rows per shard")
    ap.add_argument("--dim", type=int, default=128)
    ap.add_argument("--shards", default="2,4")
    ap.add_argument("--devices", type=int, default=1)
    ap.add_argument("--nq", type=int, default=10_000)
    ap.add_argument("--limit", type=int, default=10)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="")
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile
    from turdb_b200 import datasets as ds
    from turdb_b200.sql_operator import ShardedVectorScanBatch, VectorOp, VectorScanBatch

    if not torch.cuda.is_available():
        sys.exit("shards_sql_probe needs a CUDA device")
    counts = [int(s) for s in args.shards.split(",")]
    total = args.rows * max(counts)
    x = ds.clustered(total, args.dim, seed=1, corpus_n=total)
    ids = np.arange(total, dtype=np.uint64)
    rng = np.random.default_rng(2)
    q = (x[rng.integers(0, total, args.nq)] + 0.05 * rng.standard_normal((args.nq, args.dim), dtype=np.float32)).astype(np.float32)
    rec = dict(probe="shards_sql_probe", card=card(), rows_per_shard=args.rows, dim=args.dim, nq=args.nq, limit=args.limit,
               devices=args.devices, statement="ORDER BY emb <-> literal LIMIT %d" % args.limit, runs=[])

    def flush():
        if args.out:
            with open(args.out, "w") as f:
                json.dump(rec, f, indent=1)
        print(json.dumps(rec["runs"][-1]), flush=True)

    for S in counts:
        n = args.rows * S
        shards = [table_index(x[s * args.rows:(s + 1) * args.rows], ids[s * args.rows:(s + 1) * args.rows], s % args.devices)
                  for s in range(S)]
        one = table_index(x[:n], ids[:n])
        sharded = ShardedVectorScanBatch(shards, VectorOp.L2Distance, args.limit)
        single = VectorScanBatch(one, VectorOp.L2Distance, args.limit)
        a, b = sharded.execute(q), single.execute(q)  # warm-up (16-bit copies, modules)
        same = all(np.array_equal(u.view(np.uint8), v.view(np.uint8)) for u, v in zip(a, b))
        t_sh, t_one = [], []
        for _ in range(args.reps):
            for fn, t in ((sharded.execute, t_sh), (single.execute, t_one)):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fn(q)
                t.append((time.perf_counter() - t0) * 1e3)
        fallbacks = verbose_fallbacks(lambda: sharded.execute(q))
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            sharded.execute(q)
        kern = [e for e in prof.events() if e.device_type.name == "CUDA"]
        relay = [e for e in kern if "sql_relay" in e.name]
        first_relay = min(e.time_range.start for e in relay)
        before = [e for e in kern if e.time_range.end <= first_relay and "Memcpy" not in e.name and "Memset" not in e.name]
        filt_ms = (max(e.time_range.end for e in before) - min(e.time_range.start for e in before)) / 1e3 if before else None
        relay_ms = (max(e.time_range.end for e in relay) - first_relay) / 1e3
        per_kernel = {}
        for e in kern:
            k = re.sub(r"<.*", "", e.name.split("(")[0])
            per_kernel[k] = per_kernel.get(k, 0.0) + (e.time_range.end - e.time_range.start) / 1e3
        rec["runs"].append(dict(
            shards=S, rows=n, bit_identical_to_one_index=bool(same),
            sharded_ms_median=float(np.median(t_sh)), sharded_ms_min=float(np.min(t_sh)),
            one_index_ms_median=float(np.median(t_one)), one_index_ms_min=float(np.min(t_one)),
            statements_per_s_sharded=args.nq / (np.median(t_sh) / 1e3), statements_per_s_one_index=args.nq / (np.median(t_one) / 1e3),
            profiled_filter_span_ms=filt_ms, profiled_relay_span_ms=relay_ms, fallback_per_shard=fallbacks,
            profiled_kernel_ms={k: round(v, 4) for k, v in sorted(per_kernel.items(), key=lambda kv: -kv[1])[:16]}))
        flush()
        for s in shards:
            s.close()
        one.close()


if __name__ == "__main__":
    main()
