"""Host-side mirror of TurDB's `src/hnsw` search interface over libturdb_cuda.so.

Names, argument meaning and error behaviour follow the reference (kahflane/TurDB):
  - `DistanceFunction`           src/hnsw/mod.rs:129-137
  - `SearchResult`               src/hnsw/mod.rs:201-206
  - `HnswSearchContext`          src/hnsw/search.rs:193-225 (only ef_search survives: the heaps and the
                                 visited set live in the kernel's shared memory)
  - `CudaHnswIndex.search`       PersistentHnswIndex::search, src/hnsw/mod.rs:1092-1174
  - `CudaHnswIndex.search_filtered`  src/hnsw/mod.rs:1176-1273

Everything here is plumbing around the C ABI (include/turdb_cuda.h); there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import enum
from dataclasses import dataclass

import numpy as np

from . import _lib

INVALID_NODE = 0xFFFFFFFF
INVALID_ROW = 0xFFFFFFFFFFFFFFFF
MAX_L0_NEIGHBORS = 32
MAX_LEVEL_NEIGHBORS = 16

STATS_DTYPE = np.dtype([("n_dist", "<u4"), ("n_dist_upper", "<u4"), ("n_expanded", "<u4"), ("n_upper_hops", "<u4")])


class DistanceFunction(enum.IntEnum):
    L2 = 0
    Cosine = 1
    InnerProduct = 2


class TurdbCudaError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"turdb_cuda status {status}: {message}")
        self.status = status


def _check(rc: int):
    if rc == _lib.OK:
        return
    msg = _lib.last_error()
    if rc in (_lib.ERR_DIMENSION_MISMATCH, _lib.ERR_INVALID_ARGUMENT):
        raise ValueError(msg)
    raise TurdbCudaError(rc, msg)


@dataclass(frozen=True)
class SearchResult:
    node_id: int
    row_id: int
    distance: float


class HnswSearchContext:
    """Per-thread search context (src/hnsw/search.rs:193-225)."""

    def __init__(self, ef_search: int, max_nodes: int = 0):
        self._ef_search = int(ef_search)
        self.max_nodes = int(max_nodes)

    def ef_search(self) -> int:
        return self._ef_search

    def set_ef_search(self, ef: int) -> None:
        self._ef_search = int(ef)


def _ptr(a, t):
    return None if a is None else a.ctypes.data_as(C.POINTER(t))


class CudaHnswIndex:
    """A flattened HNSW graph resident on one B200 (device arena + fixed-stride adjacency)."""

    def __init__(self, handle, dim: int, n: int, metric: DistanceFunction, device: int, build_params=None):
        self._h = handle
        self.dim = dim
        self.n = n
        self._metric = DistanceFunction(metric)
        self.device = device
        # (m, ef_construction, mode) that `insert` uses when its arguments are omitted; None: they must be given
        self._build_params = build_params

    # ---- construction -------------------------------------------------------------------
    @classmethod
    def from_graph(cls, graph: dict, device: int = 0, metric: DistanceFunction = DistanceFunction.L2):
        """`graph`: vectors[n,dim] f32, row_ids[n] u64, levels[n] u8, l0_adj[n,32] u32, l0_cnt[n] u8,
        up_base[n] u32, up_adj[slots,16] u32, up_cnt[slots] u8, entry, max_level."""
        L = _lib.load()
        vec = np.ascontiguousarray(graph["vectors"], dtype=np.float32)
        n, dim = (vec.shape if vec.ndim == 2 else (0, int(graph.get("dim", 0))))
        keep = dict(
            vec=vec,
            row_ids=np.ascontiguousarray(graph["row_ids"], dtype=np.uint64),
            levels=np.ascontiguousarray(graph["levels"], dtype=np.uint8),
            l0_adj=np.ascontiguousarray(graph["l0_adj"], dtype=np.uint32),
            l0_cnt=np.ascontiguousarray(graph["l0_cnt"], dtype=np.uint8),
            up_base=np.ascontiguousarray(graph["up_base"], dtype=np.uint32),
            up_adj=np.ascontiguousarray(graph["up_adj"], dtype=np.uint32),
            up_cnt=np.ascontiguousarray(graph["up_cnt"], dtype=np.uint8),
        )
        g = _lib.Graph()
        g.dim = dim
        g.max_level = int(graph["max_level"])
        g.n = n
        g.entry = int(graph["entry"]) if n else INVALID_NODE
        g.vectors = _ptr(keep["vec"], C.c_float)
        g.row_ids = _ptr(keep["row_ids"], C.c_uint64)
        g.levels = _ptr(keep["levels"], C.c_uint8)
        g.l0_adj = _ptr(keep["l0_adj"], C.c_uint32)
        g.l0_cnt = _ptr(keep["l0_cnt"], C.c_uint8)
        g.up_base = _ptr(keep["up_base"], C.c_uint32)
        g.n_up_slots = int(keep["up_cnt"].shape[0])
        g.up_adj = _ptr(keep["up_adj"], C.c_uint32) if g.n_up_slots else None
        g.up_cnt = _ptr(keep["up_cnt"], C.c_uint8) if g.n_up_slots else None
        h = C.c_void_p()
        _check(L.turdb_cuda_index_create(C.byref(g), device, C.byref(h)))
        return cls(h, dim, n, metric, device)

    @classmethod
    def build(cls, vectors, row_ids=None, random_values=None, m: int = 16, ef_construction: int = 100, mode: int = 1,
              max_batch: int = 4096, device: int = 0, metric: DistanceFunction = DistanceFunction.L2, seed: int = 1234):
        """Build the graph ON THE DEVICE by the reference's insert path (insert_with_callback, src/hnsw/mod.rs:999-1084;
        turdb_cuda_index_build).  mode 0 verbatim / 1 reference-intent; max_batch = 1 is the reference's sequential
        procedure exactly.  random_values: the (0, 1] stream select_level draws from (default: seeded like the oracle's)."""
        vec = np.ascontiguousarray(vectors, dtype=np.float32)
        n, dim = vec.shape
        rid = np.arange(n, dtype=np.uint64) if row_ids is None else np.ascontiguousarray(row_ids, dtype=np.uint64)
        rnd = (1.0 - np.random.default_rng(seed).random(n)) if random_values is None else np.ascontiguousarray(random_values, np.float64)
        bp = _lib.BuildParams(dim, m, ef_construction, mode, max_batch, 0)
        h = C.c_void_p()
        _check(_lib.load().turdb_cuda_index_build(C.byref(bp), n, _ptr(vec, C.c_float), _ptr(rid, C.c_uint64),
                                                  _ptr(rnd, C.c_double), device, C.byref(h)))
        return cls(h, dim, n, metric, device, build_params=(m, ef_construction, mode))

    def insert(self, vectors, row_ids, random_values, m: int | None = None, ef_construction: int | None = None,
               mode: int | None = None, max_batch: int = 4096):
        """Append rows by the insert path (turdb_cuda_index_insert): PersistentHnswIndex::insert_with_callback for each
        row in order, new node ids self.n .. self.n + len - 1.  row_ids and random_values (the (0, 1] draw select_level
        uses) come from the caller, as in the reference's DML hook.  m / ef_construction / mode default to those of
        `build` (or of the `.hnsw` header for HnswFile.upload, mode 1).  A writer call: no other call may use this index
        while it runs.  Raises ValueError before touching the device on bad shapes, dtypes or parameters."""
        vec = np.asarray(vectors)
        if vec.dtype.kind != "f" or vec.ndim != 2 or vec.shape[1] != self.dim:
            raise ValueError(f"vectors must be float [n, {self.dim}], got {vec.dtype} {vec.shape}")
        n = vec.shape[0]
        if row_ids is None or random_values is None:
            raise ValueError("row_ids and random_values are required (one per inserted row)")
        rid = np.asarray(row_ids)
        rnd = np.asarray(random_values)
        if rid.dtype.kind not in "ui" or rid.shape != (n,):
            raise ValueError(f"row_ids must be integer [{n}], got {rid.dtype} {rid.shape}")
        if rid.dtype.kind == "i" and n and rid.min() < 0:
            raise ValueError("row_ids must be non-negative")
        if rnd.dtype.kind != "f" or rnd.shape != (n,):
            raise ValueError(f"random_values must be float [{n}], got {rnd.dtype} {rnd.shape}")
        if None in (m, ef_construction, mode):
            if self._build_params is None:
                raise ValueError("m, ef_construction and mode are required: this index was not built or read from a file")
            bm, bef, bmode = self._build_params
            m, ef_construction, mode = (bm if m is None else m, bef if ef_construction is None else ef_construction,
                                        bmode if mode is None else mode)
        vec = np.ascontiguousarray(vec, dtype=np.float32)
        rid = np.ascontiguousarray(rid, dtype=np.uint64)
        rnd = np.ascontiguousarray(rnd, dtype=np.float64)
        bp = _lib.BuildParams(self.dim, int(m), int(ef_construction), int(mode), int(max_batch), 0)
        _check(_lib.load().turdb_cuda_index_insert(self._h, C.byref(bp), n, _ptr(vec, C.c_float), _ptr(rid, C.c_uint64),
                                                   _ptr(rnd, C.c_double)))
        self.n += n

    def delete(self, node_ids) -> int:
        """Delete rows by dense node id (turdb_cuda_index_delete) and return how many nodes of the index are deleted
        after the call.  Every read path then treats them as rows the table no longer holds; node ids and the graph stay
        as they are.  Deleting a deleted node, duplicates and an empty list are allowed.  A writer call, like insert.
        Raises ValueError before touching the device on a non-integer dtype, a shape other than [n] or an id outside
        [0, node_count())."""
        ids = np.asarray(node_ids)
        if ids.ndim != 1 or (ids.size and ids.dtype.kind not in "ui"):
            raise ValueError(f"node_ids must be integer [n], got {ids.dtype} {ids.shape}")
        if ids.size and (int(ids.min()) < 0 or int(ids.max()) >= self.n):
            raise ValueError(f"node_ids must lie in [0, {self.n}), got [{int(ids.min())}, {int(ids.max())}]")
        ids = np.ascontiguousarray(ids, dtype=np.uint32)
        out = C.c_uint64(0)
        _check(_lib.load().turdb_cuda_index_delete(self._h, ids.size, _ptr(ids, C.c_uint32) if ids.size else None,
                                                   C.byref(out)))
        return int(out.value)

    def compact(self) -> np.ndarray:
        """Remove the deleted nodes (turdb_cuda_index_compact): live nodes keep their order and are renumbered 0 ..
        n_live - 1, the lists through deleted nodes are repaired, and every read path then runs as on an index that never
        had a delete.  Returns the old -> new node id map (uint32 [node count before the call]; INVALID_NODE for a
        deleted node) for rewriting the caller's NodeId map.  Without deletions: the identity map, nothing changes.  A
        writer call, like insert and delete."""
        o2n = np.zeros(max(self.n, 1), np.uint32)
        n_new = C.c_uint64(0)
        _check(_lib.load().turdb_cuda_index_compact(self._h, _ptr(o2n, C.c_uint32), C.byref(n_new)))
        o2n = o2n[:self.n]
        self.n = int(n_new.value)
        return o2n

    def export_graph(self, with_vectors: bool = True) -> dict:
        """The graph the device holds, as the flat arrays from_graph takes (turdb_cuda_index_export_graph)."""
        L = _lib.load()
        slots, entry, ml = C.c_uint64(0), C.c_uint32(0), C.c_uint32(0)
        _check(L.turdb_cuda_index_export_graph(self._h, None, None, None, None, None, None, None, None, C.byref(entry),
                                               C.byref(ml), C.byref(slots)))
        n, ns = self.n, int(slots.value)
        g = dict(vectors=np.zeros((n, self.dim), np.float32) if with_vectors else None, row_ids=np.zeros(n, np.uint64),
                 levels=np.zeros(n, np.uint8), l0_adj=np.zeros((n, 32), np.uint32), l0_cnt=np.zeros(n, np.uint8),
                 up_base=np.zeros(n, np.uint32), up_adj=np.zeros((ns, 16), np.uint32), up_cnt=np.zeros(ns, np.uint8))
        _check(L.turdb_cuda_index_export_graph(self._h, _ptr(g["vectors"], C.c_float), _ptr(g["row_ids"], C.c_uint64),
                                               _ptr(g["levels"], C.c_uint8), _ptr(g["l0_adj"], C.c_uint32),
                                               _ptr(g["l0_cnt"], C.c_uint8), _ptr(g["up_base"], C.c_uint32),
                                               _ptr(g["up_adj"], C.c_uint32) if ns else None,
                                               _ptr(g["up_cnt"], C.c_uint8) if ns else None, C.byref(entry), C.byref(ml),
                                               C.byref(slots)))
        g["entry"] = int(entry.value)
        g["max_level"] = int(ml.value)
        return g

    def close(self):
        if getattr(self, "_h", None):
            _lib.load().turdb_cuda_index_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- HnswIndex accessors (src/hnsw/mod.rs:668-724) -----------------------------------
    def dimensions(self) -> int:
        return self.dim

    def distance_fn(self) -> DistanceFunction:
        return self._metric

    def node_count(self) -> int:
        return self.n

    def info(self) -> dict:
        n, dim, ml, entry, nbytes = C.c_uint64(), C.c_uint32(), C.c_uint32(), C.c_uint32(), C.c_uint64()
        _check(_lib.load().turdb_cuda_index_info(self._h, C.byref(n), C.byref(dim), C.byref(ml), C.byref(entry),
                                                 C.byref(nbytes)))
        return dict(n=n.value, dim=dim.value, max_level=ml.value,
                    entry=None if entry.value == INVALID_NODE else entry.value, device_bytes=nbytes.value)

    def set_tuning(self, warps_per_cta: int = 0, staging_slots: int = 0, hash_bits: int = 0, segments: int = 0):
        _check(_lib.load().turdb_cuda_index_set_tuning(self._h, warps_per_cta, staging_slots, hash_bits, segments))

    def set_traversal_form(self, form: int = 0):
        """0 automatic, 1 staged (team + TMA staging), 2 direct (one warp per query); results are identical."""
        _check(_lib.load().turdb_cuda_index_set_traversal_form(self._h, form))

    def debug_counters(self, enable: bool = True):
        """Diagnostics: returns the 16 per-phase cycle counters accumulated so far and (re)arms or disarms them."""
        out = np.zeros(16, np.uint64)
        _check(_lib.load().turdb_cuda_index_debug_counters(self._h, 1 if enable else 0, _ptr(out, C.c_uint64)))
        return out

    def gather_probe(self, ctas_per_sm: int = 5, staging_slots: int = 16, cta_smem_bytes: int = 0, rounds: int = 64):
        """Diagnostics: random whole-row gather bandwidth (GB/s) at the given residency; see gather_probe.cuh."""
        ms, nbytes = C.c_float(0), C.c_uint64(0)
        _check(_lib.load().turdb_cuda_index_gather_probe(self._h, ctas_per_sm, staging_slots, cta_smem_bytes, rounds,
                                                          C.byref(ms), C.byref(nbytes)))
        return nbytes.value / ms.value / 1e6, ms.value

    def profile_begin(self, capacity: int):
        _check(_lib.load().turdb_cuda_index_profile_begin(self._h, capacity))

    def profile_read(self, capacity: int):
        """(main_ms[n], overflow_ms[n]) per-launch device times since profile_begin (sync the stream first)."""
        a = np.zeros(capacity, np.float32)
        b = np.zeros(capacity, np.float32)
        n = C.c_uint32(0)
        _check(_lib.load().turdb_cuda_index_profile_read(self._h, _ptr(a, C.c_float), _ptr(b, C.c_float), capacity,
                                                         C.byref(n)))
        return a[:n.value], b[:n.value]

    # ---- the reference's entry points ------------------------------------------------------
    def search(self, query, k: int, ctx: HnswSearchContext, metric: DistanceFunction | None = None):
        """PersistentHnswIndex::search(query, k, ctx, get_vector) -> Vec<SearchResult>."""
        rows, nodes, dist, counts, _ = self.search_batch(np.asarray(query, np.float32)[None, :], k, ctx.ef_search(),
                                                         metric)
        c = int(counts[0])
        return [SearchResult(int(nodes[0, i]), int(rows[0, i]), float(dist[0, i])) for i in range(c)]

    def search_filtered(self, query, k: int, ctx: HnswSearchContext, is_visible, row_ids=None,
                        metric: DistanceFunction | None = None):
        """search_filtered(..., is_visible: Fn(row_id) -> bool).  `row_ids` = the index's row ids (node order)."""
        if row_ids is None:
            raise ValueError("search_filtered needs the node-ordered row_ids to evaluate is_visible on the host")
        vis = visibility_bitmap(np.fromiter((bool(is_visible(int(r))) for r in row_ids), bool, len(row_ids)))
        rows, nodes, dist, counts, _ = self.search_batch(np.asarray(query, np.float32)[None, :], k, ctx.ef_search(),
                                                         metric, visible=vis)
        c = int(counts[0])
        return [SearchResult(int(nodes[0, i]), int(rows[0, i]), float(dist[0, i])) for i in range(c)]

    # ---- batched forms (what the SQL vector-scan operator and the benches call) ------------
    def search_batch(self, queries, k: int, ef: int, metric: DistanceFunction | None = None, visible=None,
                     want_stats: bool = True):
        """Host buffers in, host buffers out.  Returns (row_ids, node_ids, dist, counts, stats)."""
        q = np.ascontiguousarray(queries, dtype=np.float32)
        if q.ndim == 1:
            q = q[None, :]
        nq, qd = q.shape
        m = int(self._metric if metric is None else metric)
        kk = max(int(k), 1)
        rows = np.full((nq, kk), INVALID_ROW, np.uint64)
        nodes = np.full((nq, kk), INVALID_NODE, np.uint32)
        dist = np.full((nq, kk), np.inf, np.float32)
        counts = np.zeros(nq, np.uint32)
        stats = np.zeros(nq, STATS_DTYPE) if want_stats else None
        vis = None if visible is None else np.ascontiguousarray(visible, dtype=np.uint64)
        rc = _lib.load().turdb_cuda_search_batch(
            self._h, _ptr(q, C.c_float), qd, nq, int(k), int(ef), m, _ptr(vis, C.c_uint64), _ptr(rows, C.c_uint64),
            _ptr(nodes, C.c_uint32), _ptr(dist, C.c_float), _ptr(counts, C.c_uint32),
            None if stats is None else stats.ctypes.data_as(C.POINTER(_lib.SearchStats)))
        _check(rc)
        return rows[:, :k], nodes[:, :k], dist[:, :k], counts, stats

    def search_batch_device(self, d_queries, nq: int, k: int, ef: int, metric, d_rows, d_dist, d_counts,
                            d_nodes=0, d_stats=0, d_visible=0, stream=0):
        """Raw device addresses (ints), enqueued on `stream` (a cudaStream_t as int)."""
        m = int(self._metric if metric is None else metric)
        _check(_lib.load().turdb_cuda_search_batch_device(self._h, d_queries, self.dim, nq, k, ef, m, d_visible or None,
                                                          d_rows, d_nodes or None, d_dist, d_counts, d_stats or None,
                                                          stream or None))

    # ---- SQ8 arena (src/hnsw/quantization.rs) ----
    def enable_sq8(self, return_rows: bool = False):
        """Encode the arena as SQ8 on the device.  return_rows -> (codes u8 [n, dim], min f32 [n], scale f32 [n])."""
        L = _lib.load()
        rb = C.c_uint32(0)
        _check(L.turdb_cuda_index_enable_sq8(self._h, None, 0, C.byref(rb)))
        if not return_rows:
            return rb.value
        raw = np.zeros((self.n, rb.value), np.uint8)
        _check(L.turdb_cuda_index_enable_sq8(self._h, _ptr(raw, C.c_uint8), raw.size, C.byref(rb)))
        tail = (self.dim + 3) & ~3
        ms = raw[:, tail:tail + 8].copy().view(np.float32)
        return raw[:, :self.dim].copy(), ms[:, 0].copy(), ms[:, 1].copy()

    def search_batch_sq8_device(self, d_queries, nq: int, k: int, ef: int, metric, d_rows, d_dist, d_counts, d_nodes=0,
                                d_stats=0, stream=0, d_visible=0):
        m = int(self._metric if metric is None else metric)
        _check(_lib.load().turdb_cuda_search_batch_sq8_device(self._h, d_queries, self.dim, nq, k, ef, m, d_visible or None,
                                                              d_rows, d_nodes or None, d_dist, d_counts, d_stats or None,
                                                              stream or None))

    def bruteforce_topk(self, queries, k: int, metric: DistanceFunction | None = None, rerank_factor: int = 0):
        """Exact path: ORDER BY <distance> LIMIT k over the whole arena (src/sql/executor.rs:2239-2392)."""
        q = np.ascontiguousarray(queries, dtype=np.float32)
        if q.ndim == 1:
            q = q[None, :]
        nq, qd = q.shape
        m = int(self._metric if metric is None else metric)
        kk = max(int(k), 1)
        rows = np.full((nq, kk), INVALID_ROW, np.uint64)
        nodes = np.full((nq, kk), INVALID_NODE, np.uint32)
        dist = np.full((nq, kk), np.inf, np.float32)
        counts = np.zeros(nq, np.uint32)
        _check(_lib.load().turdb_cuda_bruteforce_topk(self._h, _ptr(q, C.c_float), qd, nq, int(k), m, int(rerank_factor),
                                                      _ptr(rows, C.c_uint64), _ptr(nodes, C.c_uint32),
                                                      _ptr(dist, C.c_float), _ptr(counts, C.c_uint32)))
        return rows[:, :k], nodes[:, :k], dist[:, :k], counts

    def bruteforce_topk_device(self, d_queries, nq: int, k: int, metric, rerank_factor: int, d_rows, d_dist,
                               d_counts, d_nodes=0, stream=0):
        m = int(self._metric if metric is None else metric)
        _check(_lib.load().turdb_cuda_bruteforce_topk_device(self._h, d_queries, self.dim, nq, k, m, rerank_factor,
                                                             d_rows, d_nodes or None, d_dist, d_counts, stream or None))


def shards_search_batch(shards, queries, k: int, ef: int, metric: DistanceFunction = DistanceFunction.L2):
    """Single-process sharded search (turdb_cuda_shards_search_batch): `shards` = list of CudaHnswIndex (one
    sub-index per GPU), replicated queries, device-to-device gather into shard 0, merge by (distance, row_id)."""
    q = np.ascontiguousarray(queries, dtype=np.float32)
    if q.ndim == 1:
        q = q[None, :]
    nq, qd = q.shape
    handles = (C.c_void_p * len(shards))(*[s._h for s in shards])
    rows = np.full((nq, k), INVALID_ROW, np.uint64)
    dist = np.full((nq, k), np.inf, np.float32)
    counts = np.zeros(nq, np.uint32)
    _check(_lib.load().turdb_cuda_shards_search_batch(handles, len(shards), _ptr(q, C.c_float), qd, nq, int(k), int(ef),
                                                      int(metric), _ptr(rows, C.c_uint64), _ptr(dist, C.c_float),
                                                      _ptr(counts, C.c_uint32)))
    return rows, dist, counts


def visibility_bitmap(visible_mask) -> np.ndarray:
    """bool[n] (node order) -> u64 bitmap, bit i of word i/64."""
    v = np.asarray(visible_mask, dtype=bool)
    n = v.shape[0]
    words = (n + 63) // 64
    padded = np.zeros(words * 64, dtype=np.uint8)
    padded[:n] = v
    return np.packbits(padded.reshape(words, 64), axis=1, bitorder="little").view(np.uint64).reshape(words)


def merge_topk_packed_device(device: int, d_gathered, shard_stride_bytes: int, n_shards: int, nq: int, k: int, d_out_rows,
                             d_out_dist, d_out_counts, stream=0):
    """Merge over one packed block per shard (rows | distances | counts): the output of a single all-gather."""
    _check(_lib.load().turdb_cuda_merge_topk_packed_device(device, d_gathered, shard_stride_bytes, n_shards, nq, k, d_out_rows,
                                                           d_out_dist, d_out_counts, stream or None))


def merge_topk_device(device: int, d_rows, d_dist, d_counts, n_shards: int, nq: int, k: int, d_out_rows, d_out_dist,
                      d_out_counts, stream=0):
    """Per-shard top-k lists [n_shards][nq][k] (the all-gather output) -> global top-k."""
    _check(_lib.load().turdb_cuda_merge_topk_device(device, d_rows, d_dist, d_counts, n_shards, nq, k, d_out_rows,
                                                    d_out_dist, d_out_counts, stream or None))
