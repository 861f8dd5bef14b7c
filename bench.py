#!/usr/bin/env python
"""bench.py — batched ANN QPS of the TurDB HNSW search hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]          # this repo's CUDA path
    python bench.py --impl reference [...]                        # the reference algorithm on host cores
    python bench.py [...] --dump-outputs DIR                      # also save the last timed step's results (.npy)

Workload at N=1 = BASELINE.json configs[1]: 1M x 384 cosine (L2-normalised synthetic embeddings),
M=16, ef_search=128, k=10, batch 10k queries.  A "step" = one batch through
turdb_cuda_search_batch_device (value; inputs resident in HBM) or through turdb_cuda_search_batch with
pinned host buffers (e2e; H2D + D2H inside the timed region).  N>1: one process per GPU, one 1M x 384
sub-index per rank (weak scaling), queries replicated, per-shard top-k all-gathered over NCCL and merged
on every rank; value = sub-index searches per second summed over ranks (= N x global QPS; unit says so at N>1).
The graph is built on the device by the reference's insert path (turdb_cuda_index_build, --graph insert); --graph knn
selects round 1's exact-kNN stand-in builder for comparison.

Only the cpu_baseline leg and --impl reference execute oracle/ (as the CPU baseline being timed, and as
the parity checker); the measured GPU path never touches it.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC_NAME = "batched ANN QPS @ recall@10>=0.95 (1M x 384 cosine, ef=128, k=10, batch 10k)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n", type=int, default=1_000_000, help="rows per GPU")
    ap.add_argument("--dim", type=int, default=384)
    ap.add_argument("--nq", type=int, default=10_000)
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--ef", type=int, default=128)
    ap.add_argument("--m", type=int, default=16)
    ap.add_argument("--latent", type=int, default=16)
    ap.add_argument("--seed", type=int, default=20261018)
    ap.add_argument("--cpu-sample", type=int, default=0, help="queries in the CPU baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--tuning", default="", help="warps,slots,hash_bits override")
    ap.add_argument("--graph", default="insert", choices=["insert", "knn"],
                    help="insert: the reference's insert path on the device (turdb_cuda_index_build); knn: exact-kNN stand-in")
    ap.add_argument("--ef-construction", type=int, default=100)
    ap.add_argument("--build-batch", type=int, default=4096, help="insert path: nodes per step (1 = sequential)")
    ap.add_argument("--build-graph-only", default="", help="(internal) build rank 0's graph, save it as .npz, exit")
    ap.add_argument("--out", default="")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the results of the last timed step as DIR/<name>.npy (float32/float64; ids -1 = none)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return args


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, arrays: dict, seed: int) -> None:
    """Writes each array (first axis = query) as <out_dir>/<name>.npy: float32 stays float32, everything else becomes
    float64 (exact for ids and counters below 2**53).  query_index.npy names the queries written: all of them, or a fixed
    seeded sample when the arrays together exceed DUMP_LIMIT_BYTES."""
    nq = len(next(iter(arrays.values())))
    out = {"query_index": np.arange(nq, dtype=np.float64)}
    out.update({k: v if v.dtype == np.float32 else v.astype(np.float64) for k, v in arrays.items()})
    total = sum(v.nbytes for v in out.values())
    if total > DUMP_LIMIT_BYTES:
        keep = np.sort(np.random.default_rng(seed).choice(nq, nq * DUMP_LIMIT_BYTES // total, replace=False))
        out = {k: v[keep] for k, v in out.items()}
    os.makedirs(out_dir, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def mark(self):
        """Samples before this point (warm-up) are discarded."""
        self.lines = []

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for nm, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def make_data(args, rank: int):
    from turdb_b200 import datasets as ds
    x = ds.gaussian_latent(args.n, args.dim, seed=args.seed + 1000 * (rank + 1), latent=args.latent, normalise=True)
    nb = 4  # distinct query batches rotated across steps
    q = ds.gaussian_latent(args.nq * nb, args.dim, seed=args.seed + 7, latent=args.latent, normalise=True)
    return x, q.reshape(nb, args.nq, args.dim)


def workload_string(args) -> str:
    """Identical in both arms (the driver compares them)."""
    return f"{args.n}x{args.dim} cosine per GPU, M={args.m}, ef={args.ef}, k={args.k}, batch {args.nq}"


def unit_string(world: int) -> str:
    return "queries/s" if world == 1 else "sub-index searches/s (N x global queries/s)"


def build_index(args, x, row_ids, device_index: int):
    """-> (CudaHnswIndex, graph arrays for the oracle, provenance string)."""
    from turdb_b200.hnsw import CudaHnswIndex, DistanceFunction
    if args.graph == "insert":
        idx = CudaHnswIndex.build(x, row_ids, None, m=args.m, ef_construction=args.ef_construction, mode=1,
                                  max_batch=args.build_batch, device=device_index, metric=DistanceFunction.Cosine, seed=args.seed)
        prov = (f"device insert path (insert_with_callback semantics, reference-intent back-links, efC={args.ef_construction}, "
                f"steps of <= {args.build_batch} nodes)")
        return idx, None, prov
    import torch
    from turdb_b200.graph_build import build_graph
    arrays = build_graph(x, m=args.m, seed=args.seed, device=torch.device("cuda", device_index))
    arrays["row_ids"] = row_ids
    idx = CudaHnswIndex.from_graph(arrays, device=device_index, metric=DistanceFunction.Cosine)
    return idx, arrays, arrays["provenance"]


def algorithmic_bytes(stats: np.ndarray, dim: int, k: int) -> int:
    """SURVEY.md §8d: n_dist*dim*4 + n_expanded*(32*4+1) + n_upper_hops*(16*4+1) + dim*4 + k*12 per query."""
    s = stats.astype(np.int64)
    return int((s[:, 0] * dim * 4 + s[:, 2] * 129 + s[:, 3] * 65 + dim * 4 + k * 12).sum())


def recall_at_k(found: np.ndarray, truth: np.ndarray) -> float:
    return float(np.mean([len(set(found[i].tolist()) & set(truth[i].tolist())) / truth.shape[1]
                          for i in range(truth.shape[0])]))


def exact_ground_truth(x_dev, q_np, k, torch):
    """Exact top-k by cosine (== L2 on normalised rows) for recall reporting; FP32 matmul, chunked."""
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    out = []
    q = torch.from_numpy(q_np).to(x_dev.device)
    for s in range(0, q.shape[0], 1024):
        sc = q[s:s + 1024] @ x_dev.T
        out.append(torch.topk(sc, k, dim=1).indices.cpu().numpy())
    torch.backends.cuda.matmul.allow_tf32 = prev
    return np.concatenate(out, 0)


# ---------------------------------------------------------------------------------------------------
def run_reference(args, rank, world):
    """The reference algorithm (oracle port, AVX2+FMA, all host threads) on the same config."""
    if rank != 0:
        return
    from oracle import binding as ob
    x, qb = make_data(args, 0)
    # The SAME graph as the GPU arm's rank 0 (same data, same seed, same builder).  Building it is not the timed path and
    # happens in a CHILD process (bench.py --build-graph-only), so that this process — the one being timed — loads the
    # oracle library and nothing of this repo's CUDA code.
    import tempfile
    path = os.path.join(tempfile.gettempdir(), f"turdb_ref_graph_{os.getpid()}.npz")
    child = [sys.executable, os.path.abspath(__file__), "--build-graph-only", path] + [a for a in sys.argv[1:] if a not in ("--impl", "reference")]
    rc = subprocess.run(child, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if rc.returncode == 0 and os.path.exists(path):
        z = np.load(path, allow_pickle=False)
        arrays = {k: z[k] for k in ("row_ids", "levels", "l0_adj", "l0_cnt", "up_base", "up_adj", "up_cnt")}
        arrays["entry"], arrays["max_level"] = int(z["entry"]), int(z["max_level"])
        prov = str(z["provenance"])
        os.remove(path)
        arrays["vectors"] = x
        g = ob.OracleGraph.from_arrays(arrays)
    elif args.n <= 50_000:  # no device to build on: the oracle's own sequential insert path (small corpora only)
        g = ob.OracleGraph.build(x, m=args.m, ef_construction=args.ef_construction, mode=ob.BUILD_INTENT, seed=args.seed)
        prov = "oracle sequential insert path (reference-intent)"
    else:
        print(json.dumps({"impl": "reference", "unavailable": "graph build child failed: " + rc.stdout[-300:].replace("\n", " ")}), flush=True)
        return
    cores = os.cpu_count() or 1
    sample = args.cpu_sample or min(args.nq, max(256, 125 * cores))
    times = []
    for it in range(args.warmup + args.steps):
        q = qb[it % qb.shape[0]][:sample]
        t = time.perf_counter()
        res = g.search(q, args.k, args.ef, ob.COSINE, n_threads=cores)
        dt = time.perf_counter() - t
        if it >= args.warmup:
            times.append(dt)
    if args.dump_outputs:
        r_rows, r_nodes, r_dist, r_cnt, r_st = res
        dump_outputs(args.dump_outputs, {"rows": r_rows.view(np.int64), "distances": r_dist, "counts": r_cnt,
                                         "nodes": r_nodes.view(np.int32),
                                         "stats": np.stack([r_st[f] for f in r_st.dtype.names], axis=1)}, args.seed)
    ms = float(np.mean(times) * 1e3)
    qps = sample / (ms / 1e3)
    line = {
        "impl": "reference", "metric": METRIC_NAME, "value": qps, "unit": unit_string(world), "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_string(args),
                   "generator": f"gaussian_latent(latent={args.latent}, normalised)", "seed": args.seed,
                   "graph": prov},
        "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": cores, "kind": "port",
                         "sample": f"{sample} of the {args.nq}-query batch per step, oracle C++ port (AVX2+FMA), {cores} threads"},
        "e2e": {"value": qps, "unit": unit_string(world), "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.build_graph_only:  # child of the reference arm: rank 0's graph -> .npz
        x, _ = make_data(args, 0)
        bidx, arrays, prov = build_index(args, x, np.arange(args.n, dtype=np.uint64), 0)
        if arrays is None:
            arrays = bidx.export_graph(with_vectors=False)
        bidx.close()
        np.savez(args.build_graph_only, provenance=np.array(prov), entry=np.array(arrays["entry"]), max_level=np.array(arrays["max_level"]),
                 **{k: arrays[k] for k in ("row_ids", "levels", "l0_adj", "l0_cnt", "up_base", "up_adj", "up_cnt")})
        return
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from turdb_b200 import _lib
    from turdb_b200.hnsw import DistanceFunction, merge_topk_packed_device
    from turdb_b200.sharding import ShardedSearch

    _lib.load()  # fail loudly if the CUDA library is missing
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import datetime
        # a mismatched collective must fail in minutes, not hold the box for NCCL's default 10
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=240))

    t0 = time.time()
    x, qb = make_data(args, rank)
    t_data = time.time() - t0
    t0 = time.time()
    # shard-local row ids are offset so the merged result names global rows
    row_ids = np.arange(args.n, dtype=np.uint64) + np.uint64(rank) * np.uint64(args.n)
    idx, arrays, provenance = build_index(args, x, row_ids, local_rank)
    torch.cuda.synchronize()
    t_build = time.time() - t0
    if args.tuning:
        idx.set_tuning(*[int(v) for v in args.tuning.split(",")])

    nb, nq, k, ef = qb.shape[0], args.nq, args.k, args.ef
    dq = torch.from_numpy(qb).to(dev)  # [nb][nq][dim] resident in HBM
    nodes = torch.empty((nq, k), dtype=torch.int32, device=dev)
    stats = torch.empty((nq, 4), dtype=torch.int32, device=dev)
    m_rows = torch.empty((nq, k), dtype=torch.int64, device=dev)
    m_dd = torch.empty((nq, k), dtype=torch.float32, device=dev)
    m_cnt = torch.empty(nq, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    launches_per_step = 2 + (1 if world > 1 else 0)  # traversal + overflow pass (+ merge)

    def local_search(dq_batch, o_rows=None, o_dd=None, o_cnt=None):
        o_rows, o_dd, o_cnt = (rows, dd, cnt) if o_rows is None else (o_rows, o_dd, o_cnt)
        idx.search_batch_device(dq_batch.data_ptr(), nq, k, ef, DistanceFunction.Cosine, o_rows.data_ptr(),
                                o_dd.data_ptr(), o_cnt.data_ptr(), nodes.data_ptr(), stats.data_ptr(), 0,
                                torch.cuda.current_stream().cuda_stream)

    def merge(gathered, block_bytes):  # ONE all-gather delivered [world][rows | distances | counts]
        merge_topk_packed_device(local_rank, gathered.data_ptr(), block_bytes, world, nq, k, m_rows.data_ptr(),
                                 m_dd.data_ptr(), m_cnt.data_ptr(), torch.cuda.current_stream().cuda_stream)
        return m_rows, m_dd, m_cnt

    sharded = ShardedSearch(dist, world, local_search, merge, nq, k, dev)
    rows, dd, cnt = sharded.rows, sharded.dd, sharded.cnt  # the rank's own top-k lives inside its packed block

    def step(i):
        return sharded.search_batch(dq[i % nb])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- value: device-resident inputs ----
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.5)  # nvidia-smi needs a moment before its first sample
    for i in range(args.warmup):
        step(i)
    barrier()
    if rank == 0:
        sampler.mark()
    prof_steps = min(args.steps, 4096)  # the index keeps per-launch times of at most 4096 launches
    idx.profile_begin(prof_steps)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(args.steps):
        last = step(args.warmup + i)
    e1.record()
    barrier()
    elapsed_ms = e0.elapsed_time(e1)
    kern_ms, over_ms = idx.profile_read(prof_steps)
    if args.dump_outputs and rank == 0:  # copied now: the work below reuses these buffers
        l_rows, l_dd, l_cnt = (t.cpu().numpy() for t in last)
        dump_outputs(args.dump_outputs, {"rows": l_rows, "distances": l_dd, "counts": l_cnt,
                                         "nodes": nodes.cpu().numpy(), "stats": stats.cpu().numpy()}, args.seed)
    if rank == 0 and elapsed_ms < 400:  # keep the GPU under the same load until the sampler has a few readings
        # rank-local kernel launches only: a collective here would not be matched by the other ranks
        t_end = time.time() + 0.45
        i = 0
        while time.time() < t_end:
            local_search(dq[i % nb])
            i += 1
        torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    if world > 1:
        t = torch.tensor([elapsed_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms = float(t.item())
    ms_per_step = elapsed_ms / args.steps
    value = world * nq / (ms_per_step / 1e3)

    # per-launch algorithmic bytes: counters of each distinct batch (identical to the oracle's, see tests)
    batch_bytes = []
    for b in range(nb):
        step(b)
        torch.cuda.synchronize()
        batch_bytes.append(algorithmic_bytes(stats.cpu().numpy(), args.dim, k))
    step_bytes = [batch_bytes[(args.warmup + i) % nb] for i in range(len(kern_ms))]
    achieved = float(np.sum(step_bytes) / (np.sum(kern_ms) / 1e3) / 1e9)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    # DRAM bytes of one traversal launch from the committed `ncu --set full` capture of this kernel on this
    # workload (profiles/): read + write, per launch like `achieved`'s numerator
    traffic, traffic_src = None, None
    try:
        import glob
        cands = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_traffic_hnsw_search_1m384.json")))
        if cands and args.n == 1_000_000 and args.dim == 384 and args.ef == 128 and args.nq == 10_000:
            tj = json.load(open(cands[-1]))
            traffic, traffic_src = float(tj["dram_bytes_per_launch"]), os.path.relpath(cands[-1], ROOT)
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_kind = "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)"

    # ---- e2e: host buffers through the public C-ABI call, pinned memory, H2D + D2H inside ----
    hq = [torch.from_numpy(qb[b]).pin_memory() for b in range(nb)]
    h_rows = torch.empty((nq, k), dtype=torch.int64).pin_memory()
    h_dd = torch.empty((nq, k), dtype=torch.float32).pin_memory()
    h_cnt = torch.empty(nq, dtype=torch.int32).pin_memory()
    L = _lib.load()
    import ctypes as C

    # N>1: the step is H2D of the query batch -> per-shard search -> ONE NCCL all-gather -> merge -> D2H of the merged
    # top-k.  One caller per rank (the collective must be issued in one order on all ranks), but the copies run on a
    # copy stream, double-buffered: batch i+1 goes up and result i-1 comes down while batch i is searched.
    copy_stream = torch.cuda.Stream(device=dev)
    dq_e2e = [torch.empty((nq, args.dim), dtype=torch.float32, device=dev) for _ in range(2)]
    res_dev = [(torch.empty_like(m_rows), torch.empty_like(m_dd), torch.empty_like(m_cnt)) for _ in range(2)]
    res_host = [(torch.empty((nq, k), dtype=torch.int64).pin_memory(), torch.empty((nq, k), dtype=torch.float32).pin_memory(),
                 torch.empty(nq, dtype=torch.int32).pin_memory()) for _ in range(2)]

    def e2e_pipeline(first, count):
        main = torch.cuda.current_stream()
        up = [torch.cuda.Event() for _ in range(2)]
        done = [torch.cuda.Event() for _ in range(2)]
        down = [torch.cuda.Event() for _ in range(2)]
        with torch.cuda.stream(copy_stream):
            dq_e2e[0].copy_(hq[first % nb], non_blocking=True)
            up[0].record(copy_stream)
        for j in range(count):
            b = j & 1
            if j + 1 < count:  # next batch goes up while this one is searched
                with torch.cuda.stream(copy_stream):
                    dq_e2e[b ^ 1].copy_(hq[(first + j + 1) % nb], non_blocking=True)
                    up[b ^ 1].record(copy_stream)
            main.wait_event(up[b])
            if j >= 2:
                main.wait_event(down[b])  # result buffer b has been read back
            sharded.search_batch(dq_e2e[b])
            for dst, src in zip(res_dev[b], (m_rows, m_dd, m_cnt)):
                dst.copy_(src, non_blocking=True)
            done[b].record(main)
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(done[b])
                for dst, src in zip(res_host[b], res_dev[b]):
                    dst.copy_(src, non_blocking=True)
                down[b].record(copy_stream)
        torch.cuda.synchronize()

    # N=1: two host threads issue alternate batches through the same call.  The ABI is re-entrant (every call owns a
    # stream and its scratch), so one caller's H2D/D2H copies overlap the other's kernel — what a multi-connection
    # host does.  N>1 keeps one caller per rank: the merge's collectives must be issued in one order on all ranks.
    e2e_callers = 2 if world == 1 else 1
    bufs = [(h_rows, h_dd, h_cnt)]
    for _ in range(e2e_callers - 1):
        bufs.append((torch.empty((nq, k), dtype=torch.int64).pin_memory(), torch.empty((nq, k), dtype=torch.float32).pin_memory(),
                     torch.empty(nq, dtype=torch.int32).pin_memory()))

    def e2e_call(i, b):
        r_, d_, c_ = bufs[b]
        rc = L.turdb_cuda_search_batch(idx._h, C.cast(hq[i % nb].data_ptr(), C.POINTER(C.c_float)), args.dim, nq, k, ef,
                                       int(DistanceFunction.Cosine), None, C.cast(r_.data_ptr(), C.POINTER(C.c_uint64)), None,
                                       C.cast(d_.data_ptr(), C.POINTER(C.c_float)), C.cast(c_.data_ptr(), C.POINTER(C.c_uint32)),
                                       None)
        assert rc == 0, _lib.last_error()

    def e2e_run(first, count):
        if e2e_callers == 1:
            e2e_pipeline(first, count)
            return
        def worker(b):
            for i in range(first + b, first + count, e2e_callers):
                e2e_call(i, b)
        ts = [threading.Thread(target=worker, args=(b,)) for b in range(e2e_callers)]
        for t_ in ts:
            t_.start()
        for t_ in ts:
            t_.join()

    e2e_run(0, args.warmup)
    barrier()
    t_start = time.perf_counter()
    e2e_run(args.warmup, args.steps)
    barrier()
    e2e_s = time.perf_counter() - t_start
    if world > 1:
        t = torch.tensor([e2e_s], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_value = world * nq * args.steps / e2e_s
    h2d = nq * args.dim * 4
    d2h = nq * k * 8 + nq * k * 4 + nq * 4

    # ---- quality: recall@10 vs exact ground truth (shard-local), and the CPU baseline on rank 0 ----
    step(0)
    torch.cuda.synchronize()
    gpu_nodes = nodes.cpu().numpy().view(np.uint32)
    gpu_dist = dd.cpu().numpy()
    # ground truth from the exact path (tensor-core pass + FP32 rerank), cross-checked below on 200 queries by
    # the CPU oracle's exact SQL scan and by an FP32 matmul
    n_gt = min(nq, 2000)
    e_rows = torch.empty((nq, k), dtype=torch.int64, device=dev)
    e_dd = torch.empty((nq, k), dtype=torch.float32, device=dev)
    e_nodes = torch.empty((nq, k), dtype=torch.int32, device=dev)
    e_cnt = torch.empty(nq, dtype=torch.int32, device=dev)
    idx.bruteforce_topk_device(dq[0].data_ptr(), nq, k, DistanceFunction.Cosine, 0, e_rows.data_ptr(), e_dd.data_ptr(),
                               e_cnt.data_ptr(), e_nodes.data_ptr(), stream)
    torch.cuda.synchronize()
    t_ex = time.perf_counter()
    idx.bruteforce_topk_device(dq[0].data_ptr(), nq, k, DistanceFunction.Cosine, 0, e_rows.data_ptr(), e_dd.data_ptr(),
                               e_cnt.data_ptr(), e_nodes.data_ptr(), stream)
    torch.cuda.synchronize()
    exact_ms = (time.perf_counter() - t_ex) * 1e3
    gt_all = e_nodes.cpu().numpy().view(np.uint32)
    gt = gt_all[:n_gt]
    recall = recall_at_k(gpu_nodes[:n_gt], gt)
    x_dev = torch.from_numpy(x).to(dev)
    gt_mm = exact_ground_truth(x_dev, qb[0][:200], k, torch)
    del x_dev
    exact_info = {"ms_per_batch": exact_ms, "tflops": 2.0 * nq * args.n * args.dim / exact_ms / 1e9,
                  "frac_of_measured_bf16_peak": (2.0 * nq * args.n * args.dim / exact_ms / 1e9) / float(peaks.get("bf16_tflops", 1655.7)),
                  "agreement_with_fp32_matmul_top10": recall_at_k(gt_all[:200], gt_mm)}

    cpu_baseline = None
    parity = None
    if rank == 0 and not args.no_cpu_baseline:
        from oracle import binding as ob
        if arrays is None:
            arrays = idx.export_graph()
        arrays["vectors"] = x
        g = ob.OracleGraph.from_arrays(arrays)
        cores = os.cpu_count() or 1
        sample = args.cpu_sample or min(nq, max(256, 125 * cores))
        g.search(qb[1][:min(sample, 256)], k, ef, ob.COSINE, n_threads=cores)  # warm-up
        reps, t_cpu = 0, 0.0
        while reps < 3 or (t_cpu < 10.0 and reps < 50):
            t = time.perf_counter()
            c_rows, c_nodes, c_dist, c_cnt, c_st = g.search(qb[0][:sample], k, ef, ob.COSINE, n_threads=cores)
            t_cpu += time.perf_counter() - t
            reps += 1
        cpu_qps = sample * reps / t_cpu
        t = time.perf_counter()
        g.search(qb[0][:min(sample, 512)], k, ef, ob.COSINE, n_threads=1)
        cpu_qps_1 = min(sample, 512) / (time.perf_counter() - t)
        same = np.array([np.array_equal(gpu_nodes[i], c_nodes[i]) for i in range(sample)])
        same_d = np.array([np.array_equal(gpu_dist[i].view(np.uint32), c_dist[i].view(np.uint32)) for i in range(sample)])
        parity = {"queries": int(sample), "id_set_match": float(same.mean()), "distance_bits_match": float(same_d.mean()),
                  "cpu_recall_at_10": recall_at_k(c_nodes[:min(sample, n_gt)], gt[:min(sample, n_gt)])}
        s_rows, _, _ = ob.sql_topk(x, qb[0][:200], k, op=ob.COSINE, n_threads=cores)  # the reference's exact SQL scan
        exact_info["agreement_with_cpu_sql_scan_top10"] = recall_at_k(gt_all[:200], s_rows.astype(np.uint32))
        cpu_baseline = {"value": cpu_qps, "unit": "queries/s", "cores": cores, "kind": "port",
                        "sample": f"{sample} queries of batch 0 x {reps} reps, oracle C++ port (AVX2+FMA, flat arrays), "
                                  f"{cores} threads; 1 thread: {cpu_qps_1:.0f} q/s"}

    if rank == 0:
        line = {
            "metric": METRIC_NAME, "value": value, "unit": unit_string(world), "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {
                "workload": workload_string(args),
                "generator": f"gaussian_latent(latent={args.latent}, normalised)", "seed": args.seed,
                "graph": provenance, "graph_build_s": round(t_build, 1), "data_gen_s": round(t_data, 1),
                "l2_policy": "inputs larger than L2 (1.5 GB arena, 4 rotating query batches)",
                "sharding": "one sub-index per GPU, queries replicated, ONE NCCL all-gather of the packed top-k + merge" if world > 1 else "single index",
                "global_qps": value / world,
            },
            "recall_at_10": recall,
            "recall_ok": bool(recall >= 0.95),  # the metric is QPS AT recall@10 >= 0.95: a record below it is not a result
            "exact_path": exact_info,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_unit": "DRAM bytes per launch (ncu dram__bytes_read.sum + dram__bytes_write.sum)",
                         "traffic_source": traffic_src, "peak_kind": peak_kind, "kernel": "hnsw_search_kernel<cosine>",
                         "kernel_ms_avg": float(np.mean(kern_ms)), "overflow_pass_ms_avg": float(np.mean(over_ms)),
                         "algorithmic_bytes_per_launch": float(np.mean(step_bytes))},
            "cpu_baseline": cpu_baseline,
            "parity": parity,
            "e2e": {"value": e2e_value, "unit": unit_string(world), "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "host_callers": e2e_callers,
                    "how": "two host threads through turdb_cuda_search_batch (pinned host buffers)" if world == 1 else
                           "one caller per rank; copies double-buffered on a copy stream around search + all-gather + merge"},
            "gpu_launches": launches_per_step * args.steps,
            "clocks": clocks,
        }
        s = json.dumps(line)
        print(s, flush=True)
        if args.out:
            open(args.out, "w").write(s + "\n")
    idx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
