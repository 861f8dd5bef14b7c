"""ctypes loader for libturdb_cuda.so.  Fails loudly: there is no CPU or PyTorch fallback."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TURDB_CUDA_LIB") or os.path.join(HERE, "libturdb_cuda.so")  # override: A/B builds

OK, ERR_INVALID_ARGUMENT, ERR_DIMENSION_MISMATCH, ERR_CUDA, ERR_OOM, ERR_UNSUPPORTED, ERR_NO_DEVICE = range(7)


class Graph(C.Structure):
    """turdb_cuda_graph (include/turdb_cuda.h)."""
    _fields_ = [("dim", C.c_uint32), ("max_level", C.c_uint32), ("n", C.c_uint64), ("entry", C.c_uint32),
                ("reserved", C.c_uint32), ("vectors", C.POINTER(C.c_float)), ("row_ids", C.POINTER(C.c_uint64)),
                ("levels", C.POINTER(C.c_uint8)), ("l0_adj", C.POINTER(C.c_uint32)), ("l0_cnt", C.POINTER(C.c_uint8)),
                ("up_base", C.POINTER(C.c_uint32)), ("up_adj", C.POINTER(C.c_uint32)), ("up_cnt", C.POINTER(C.c_uint8)),
                ("n_up_slots", C.c_uint64)]


class SearchStats(C.Structure):
    _fields_ = [("n_dist", C.c_uint32), ("n_dist_upper", C.c_uint32), ("n_expanded", C.c_uint32),
                ("n_upper_hops", C.c_uint32)]


class HnswFileInfo(C.Structure):
    """turdb_cuda_hnsw_file_info (include/turdb_cuda.h)."""
    _fields_ = [("index_id", C.c_uint64), ("table_id", C.c_uint64), ("dimensions", C.c_uint32), ("m", C.c_uint32),
                ("m0", C.c_uint32), ("ef_construction", C.c_uint32), ("ef_search", C.c_uint32),
                ("distance_fn", C.c_uint8), ("quantization", C.c_uint8), ("header_max_level", C.c_uint8),
                ("max_level", C.c_uint8), ("has_entry", C.c_uint8), ("reserved", C.c_uint8 * 3),
                ("entry", C.c_uint32), ("flags", C.c_uint32), ("n_pages", C.c_uint32), ("n_foreign_pages", C.c_uint32),
                ("n_suspect_pages", C.c_uint32), ("header_node_count", C.c_uint64), ("header_vector_count", C.c_uint64),
                ("n_nodes", C.c_uint64), ("n_tombstones", C.c_uint64), ("n_up_slots", C.c_uint64),
                ("n_deleted_slots", C.c_uint64), ("n_unreadable_slots", C.c_uint64)]


class BuildParams(C.Structure):
    _fields_ = [("dim", C.c_uint32), ("m", C.c_uint32), ("ef_construction", C.c_uint32), ("mode", C.c_uint32),
                ("max_batch", C.c_uint32), ("reserved", C.c_uint32)]


GET_VECTOR_FN = C.CFUNCTYPE(C.c_int32, C.c_void_p, C.c_uint64, C.POINTER(C.c_float))

# every symbol include/turdb_cuda.h declares
EXPORTS = [
    "turdb_cuda_abi_version", "turdb_cuda_last_error", "turdb_cuda_device_count", "turdb_cuda_index_create",
    "turdb_cuda_index_destroy", "turdb_cuda_index_info", "turdb_cuda_search_batch", "turdb_cuda_search_batch_device",
    "turdb_cuda_index_set_tuning", "turdb_cuda_index_set_traversal_form", "turdb_cuda_index_profile_begin", "turdb_cuda_index_profile_read",
    "turdb_cuda_index_debug_counters", "turdb_cuda_bruteforce_topk", "turdb_cuda_bruteforce_topk_device",
    "turdb_cuda_merge_topk_device", "turdb_cuda_merge_topk_packed_device", "turdb_cuda_index_gather_probe",
    "turdb_cuda_hnsw_file_open", "turdb_cuda_hnsw_file_open_memory", "turdb_cuda_hnsw_file_close",
    "turdb_cuda_hnsw_file_get_info", "turdb_cuda_hnsw_file_nodes", "turdb_cuda_hnsw_file_graph",
    "turdb_cuda_hnsw_file_upload", "turdb_cuda_sql_topk_batch", "turdb_cuda_sql_topk_batch_device",
    "turdb_cuda_index_enable_sq8", "turdb_cuda_search_batch_sq8_device", "turdb_cuda_shards_search_batch",
    "turdb_cuda_index_build", "turdb_cuda_index_export_graph", "turdb_cuda_index_insert",
    "turdb_cuda_sql_range_batch", "turdb_cuda_sql_range_batch_device", "turdb_cuda_sql_range_topk_batch",
    "turdb_cuda_sql_range_topk_batch_device", "turdb_cuda_index_delete", "turdb_cuda_index_compact",
    "turdb_cuda_shards_sql_topk_batch",
]

_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing. Build it with `python -m turdb_b200.build` (needs nvcc). "
            "turdb_b200 has no CPU or PyTorch fallback for the search path.")
    L = C.CDLL(LIB_PATH)
    vp, u8, u32, u64, i32 = C.c_void_p, C.c_uint8, C.c_uint32, C.c_uint64, C.c_int32
    pf, pu32, pu64, pu8 = C.POINTER(C.c_float), C.POINTER(u32), C.POINTER(u64), C.POINTER(u8)
    L.turdb_cuda_abi_version.restype = u32
    L.turdb_cuda_last_error.restype = C.c_char_p
    L.turdb_cuda_device_count.argtypes = [C.POINTER(i32)]
    L.turdb_cuda_index_create.argtypes = [C.POINTER(Graph), i32, C.POINTER(vp)]
    L.turdb_cuda_index_destroy.argtypes = [vp]
    L.turdb_cuda_index_info.argtypes = [vp, pu64, pu32, pu32, pu32, pu64]
    L.turdb_cuda_index_set_tuning.argtypes = [vp, u32, u32, u32, u32]
    L.turdb_cuda_index_set_traversal_form.argtypes = [vp, u32]
    L.turdb_cuda_index_debug_counters.argtypes = [vp, i32, pu64]
    L.turdb_cuda_index_profile_begin.argtypes = [vp, u32]
    L.turdb_cuda_index_profile_read.argtypes = [vp, pf, pf, u32, pu32]
    L.turdb_cuda_index_gather_probe.argtypes = [vp, u32, u32, u32, u32, pf, pu64]
    L.turdb_cuda_search_batch.argtypes = [vp, pf, u32, u32, u32, u32, u8, pu64, pu64, pu32, pf, pu32,
                                          C.POINTER(SearchStats)]
    # _device entries take raw device addresses
    L.turdb_cuda_search_batch_device.argtypes = [vp, vp, u32, u32, u32, u32, u8, vp, vp, vp, vp, vp, vp, vp]
    L.turdb_cuda_bruteforce_topk.argtypes = [vp, pf, u32, u32, u32, u8, u32, pu64, pu32, pf, pu32]
    L.turdb_cuda_bruteforce_topk_device.argtypes = [vp, vp, u32, u32, u32, u8, u32, vp, vp, vp, vp, vp]
    L.turdb_cuda_merge_topk_device.argtypes = [i32, vp, vp, vp, u32, u32, u32, vp, vp, vp, vp]
    L.turdb_cuda_merge_topk_packed_device.argtypes = [i32, vp, u64, u32, u32, u32, vp, vp, vp, vp]
    L.turdb_cuda_sql_topk_batch.argtypes = [vp, pf, u32, u32, u32, u32, u8, u8, i32, u32, pu64, C.POINTER(C.c_double),
                                            C.POINTER(C.c_double), pu32]
    L.turdb_cuda_sql_topk_batch_device.argtypes = [vp, vp, u32, u32, u32, u32, u8, u8, i32, u32, vp, vp, vp, vp, vp]
    L.turdb_cuda_sql_range_batch.argtypes = [vp, pf, u32, u32, u8, u8, C.POINTER(C.c_double), u32, u32, pu64,
                                             C.POINTER(C.c_double), pu32]
    L.turdb_cuda_sql_range_batch_device.argtypes = [vp, vp, u32, u32, u8, u8, vp, u32, u32, vp, vp, vp, vp]
    L.turdb_cuda_sql_range_topk_batch.argtypes = [vp, pf, u32, u32, u8, u8, C.POINTER(C.c_double), u8, u8, u32, u32, pu64,
                                                  C.POINTER(C.c_double), C.POINTER(C.c_double), pu32]
    L.turdb_cuda_sql_range_topk_batch_device.argtypes = [vp, vp, u32, u32, u8, u8, vp, u8, u8, u32, u32, vp, vp, vp, vp, vp]
    L.turdb_cuda_index_enable_sq8.argtypes = [vp, pu8, u64, pu32]
    L.turdb_cuda_search_batch_sq8_device.argtypes = [vp, vp, u32, u32, u32, u32, u8, vp, vp, vp, vp, vp, vp, vp]
    L.turdb_cuda_shards_search_batch.argtypes = [C.POINTER(vp), u32, pf, u32, u32, u32, u32, u8, pu64, pf, pu32]
    L.turdb_cuda_shards_sql_topk_batch.argtypes = [C.POINTER(vp), u32, pf, u32, u32, u32, u32, u8, u8, pu64,
                                                    C.POINTER(C.c_double), C.POINTER(C.c_double), pu32]
    L.turdb_cuda_index_build.argtypes = [C.POINTER(BuildParams), u64, pf, pu64, C.POINTER(C.c_double), i32, C.POINTER(vp)]
    L.turdb_cuda_index_insert.argtypes = [vp, C.POINTER(BuildParams), u64, pf, pu64, C.POINTER(C.c_double)]
    L.turdb_cuda_index_delete.argtypes = [vp, u64, pu32, pu64]
    L.turdb_cuda_index_compact.argtypes = [vp, pu32, pu64]
    L.turdb_cuda_index_export_graph.argtypes = [vp, pf, pu64, pu8, pu32, pu8, pu32, pu32, pu8, pu32, pu32, pu64]
    L.turdb_cuda_hnsw_file_open.argtypes = [C.c_char_p, C.POINTER(vp)]
    L.turdb_cuda_hnsw_file_open_memory.argtypes = [pu8, u64, C.POINTER(vp)]
    L.turdb_cuda_hnsw_file_close.argtypes = [vp]
    L.turdb_cuda_hnsw_file_get_info.argtypes = [vp, C.POINTER(HnswFileInfo)]
    L.turdb_cuda_hnsw_file_nodes.argtypes = [vp, pu64, pu32, C.POINTER(C.c_uint16)]
    L.turdb_cuda_hnsw_file_graph.argtypes = [vp, pf, C.POINTER(Graph)]
    L.turdb_cuda_hnsw_file_upload.argtypes = [vp, pf, pu8, GET_VECTOR_FN, vp, i32, C.POINTER(vp)]
    for name in EXPORTS:
        if name not in ("turdb_cuda_abi_version", "turdb_cuda_last_error"):
            getattr(L, name).restype = i32
    _lib = L
    return L


def last_error() -> str:
    return (load().turdb_cuda_last_error() or b"").decode("utf-8", "replace")
