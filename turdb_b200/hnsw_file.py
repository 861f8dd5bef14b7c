"""Reader of the reference's on-disk HNSW index (`.hnsw`) -> `CudaHnswIndex` (SURVEY.md §8f rank 1).

Mirrors what `PersistentHnswIndex::open` + `rebuild_row_id_map` + `read_node` see in a file
(src/hnsw/mod.rs:811-859, 906-911; layout src/hnsw/storage.rs:98-119, 322-383, 485-546): parsing is done
by libturdb_cuda.so (`csrc/hnsw_file.inl`, host code, no GPU needed); this module is the binding.
Vectors are not part of the file — the table owns them (mod.rs:1097) — so the caller passes them per
dense node id or as a `get_vector(row_id) -> Optional[sequence]` callable like the reference's closure.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from .hnsw import CudaHnswIndex, DistanceFunction, _check, _ptr

FLAG_SUSPECT_PAGES, FLAG_TOMBSTONES, FLAG_NODE_COUNT_MISMATCH, FLAG_MAX_LEVEL_CLAMPED, FLAG_TRAILING_BYTES = 1, 2, 4, 8, 16


class HnswFile:
    """A parsed `.hnsw` file (host memory)."""

    def __init__(self, handle):
        self._h = handle
        info = _lib.HnswFileInfo()
        _check(_lib.load().turdb_cuda_hnsw_file_get_info(self._h, C.byref(info)))
        self.info = {name: getattr(info, name) for name, _ in _lib.HnswFileInfo._fields_ if name != "reserved"}

    @classmethod
    def open(cls, path: str) -> "HnswFile":
        h = C.c_void_p()
        _check(_lib.load().turdb_cuda_hnsw_file_open(str(path).encode(), C.byref(h)))
        return cls(h)

    @classmethod
    def from_bytes(cls, data: bytes) -> "HnswFile":
        h = C.c_void_p()
        buf = (C.c_uint8 * len(data)).from_buffer_copy(data)
        _check(_lib.load().turdb_cuda_hnsw_file_open_memory(buf, len(data), C.byref(h)))
        return cls(h)

    def close(self):
        if getattr(self, "_h", None):
            _lib.load().turdb_cuda_hnsw_file_close(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- header mirror (HnswIndex::from_header, mod.rs:647-660) ----
    def dimensions(self) -> int:
        return self.info["dimensions"]

    def distance_fn(self) -> DistanceFunction:
        return DistanceFunction(self.info["distance_fn"])

    def ef_search(self) -> int:
        return self.info["ef_search"]

    def node_count(self) -> int:
        return self.info["n_nodes"]

    @property
    def n_total(self) -> int:
        return self.info["n_nodes"] + self.info["n_tombstones"]

    def nodes(self):
        """(row_ids u64, pages u32, slots u16) per dense id; tombstones (row_id 0) come last."""
        n = self.n_total
        rows, pages, slots = np.zeros(n, np.uint64), np.zeros(n, np.uint32), np.zeros(n, np.uint16)
        _check(_lib.load().turdb_cuda_hnsw_file_nodes(self._h, _ptr(rows, C.c_uint64), _ptr(pages, C.c_uint32),
                                                      _ptr(slots, C.c_uint16)))
        return rows, pages, slots

    def graph(self, vectors: np.ndarray | None = None) -> dict:
        """The flattened arrays (copies) in the layout `CudaHnswIndex.from_graph` and the C ABI take."""
        g = _lib.Graph()
        _check(_lib.load().turdb_cuda_hnsw_file_graph(self._h, None, C.byref(g)))
        n, slots = int(g.n), int(g.n_up_slots)

        def arr(ptr, count, dtype):
            return np.ctypeslib.as_array(ptr, shape=(count,)).astype(dtype, copy=True) if count else np.zeros(0, dtype)

        out = dict(dim=int(g.dim), max_level=int(g.max_level), entry=int(g.entry),
                   row_ids=arr(g.row_ids, n, np.uint64), levels=arr(g.levels, n, np.uint8),
                   l0_adj=arr(g.l0_adj, n * 32, np.uint32).reshape(n, 32), l0_cnt=arr(g.l0_cnt, n, np.uint8),
                   up_base=arr(g.up_base, n, np.uint32), up_adj=arr(g.up_adj, slots * 16, np.uint32).reshape(slots, 16),
                   up_cnt=arr(g.up_cnt, slots, np.uint8), provenance="hnsw-file")
        if vectors is not None:
            out["vectors"] = self._full_vectors(vectors)
        return out

    def _full_vectors(self, vectors: np.ndarray) -> np.ndarray:
        vec = np.ascontiguousarray(vectors, dtype=np.float32)
        if vec.shape != (self.info["n_nodes"], self.info["dimensions"]):
            raise ValueError(f"vectors must be [{self.info['n_nodes']}, {self.info['dimensions']}], got {vec.shape}")
        if self.info["n_tombstones"]:
            vec = np.concatenate([vec, np.full((self.info["n_tombstones"], vec.shape[1]), np.inf, np.float32)], 0)
        return vec

    def upload(self, vectors: np.ndarray | None = None, get_vector=None, present: np.ndarray | None = None,
               device: int = 0, metric: DistanceFunction | None = None) -> CudaHnswIndex:
        """Device index of this file.  `vectors` [n_nodes, dim] in dense-id order and/or `get_vector(row_id)`
        returning a sequence of `dim` floats or None (the reference's closure, mod.rs:1097)."""
        L = _lib.load()
        dim = self.info["dimensions"]
        vec_p = None
        if vectors is not None:
            vec = np.ascontiguousarray(vectors, dtype=np.float32)
            if vec.shape != (self.info["n_nodes"], dim):
                raise ValueError(f"vectors must be [{self.info['n_nodes']}, {dim}], got {vec.shape}")
            vec_p = _ptr(vec, C.c_float)
        pres_p = None
        if present is not None:
            pres = np.ascontiguousarray(present, dtype=np.uint8)
            pres_p = _ptr(pres, C.c_uint8)
        cb = C.cast(None, _lib.GET_VECTOR_FN)
        if get_vector is not None:
            def _cb(_user, row_id, out):
                v = get_vector(int(row_id))
                if v is None:
                    return 0
                a = np.asarray(v, dtype=np.float32)
                if a.shape != (dim,):
                    return 0
                C.memmove(out, a.ctypes.data, dim * 4)
                return 1
            cb = _lib.GET_VECTOR_FN(_cb)
        h = C.c_void_p()
        _check(L.turdb_cuda_hnsw_file_upload(self._h, vec_p, pres_p, cb, None, device, C.byref(h)))
        m = self.distance_fn() if metric is None else DistanceFunction(metric)
        return CudaHnswIndex(h, dim, self.n_total, m, device, build_params=(self.info["m"], self.info["ef_construction"], 1))
