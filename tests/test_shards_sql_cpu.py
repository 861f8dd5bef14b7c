"""turdb_cuda_shards_sql_topk_batch without a device: the C entry's argument checks (operators and window before the
shards, the shard array before anything else) and the Python wrapper's validation, which must reject bad input before
the library is called."""
import ctypes as C

import numpy as np
import pytest

from turdb_b200 import _lib
from turdb_b200.hnsw import CudaHnswIndex, DistanceFunction
from turdb_b200.sql_operator import ShardedVectorScanBatch, VectorOp

Q = np.zeros((3, 8), np.float32)


def entry(shards, n_shards, op=0, limit=10, offset=0, proj_op=0, project=False):
    L = _lib.load()
    size = 3 * min(max(limit, 1), 512)  # a rejected window is never written
    rows = np.zeros(size, np.uint64)
    keys = np.zeros(size)
    proj = np.zeros(size)
    cnt = np.zeros(3, np.uint32)
    d = C.POINTER(C.c_double)
    arr = None if shards is None else (C.c_void_p * max(len(shards), 1))(*shards)
    return L.turdb_cuda_shards_sql_topk_batch(arr, n_shards, Q.ctypes.data_as(C.POINTER(C.c_float)), 8, 3, limit, offset,
                                              op, proj_op, rows.ctypes.data_as(C.POINTER(C.c_uint64)), keys.ctypes.data_as(d),
                                              proj.ctypes.data_as(d) if project else None,
                                              cnt.ctypes.data_as(C.POINTER(C.c_uint32)))


@pytest.mark.parametrize("shards,n_shards", [(None, 1), ([], 0), ([None] * 33, 33)])
def test_missing_or_oversized_shard_arrays_are_invalid_arguments(shards, n_shards):
    assert entry(shards, n_shards) == _lib.ERR_INVALID_ARGUMENT
    assert b"n_shards" in _lib.load().turdb_cuda_last_error()


def test_a_null_shard_is_an_invalid_argument():
    assert entry([None, None], 2) == _lib.ERR_INVALID_ARGUMENT
    assert b"shard 0 is null" in _lib.load().turdb_cuda_last_error()


def test_order_by_inner_product_is_unsupported():
    assert entry([None], 1, op=2) == _lib.ERR_UNSUPPORTED
    assert b"<#>" in _lib.load().turdb_cuda_last_error()


@pytest.mark.parametrize("limit,offset", [(513, 0), (0, 513), (500, 13), (2**32 - 1, 1)])
def test_window_past_the_heap_limit_is_unsupported(limit, offset):
    assert entry([None], 1, limit=limit, offset=offset) == _lib.ERR_UNSUPPORTED
    assert b"limit + offset" in _lib.load().turdb_cuda_last_error()


def test_unknown_projection_is_an_invalid_argument():
    assert entry([None], 1, proj_op=3, project=True) == _lib.ERR_INVALID_ARGUMENT
    assert b"proj_op" in _lib.load().turdb_cuda_last_error()
    # without out_proj the projection operator is not read; limit + offset = 512 passes: the shard is null
    assert entry([None], 1, limit=500, offset=12, proj_op=3) == _lib.ERR_INVALID_ARGUMENT
    assert b"shard 0 is null" in _lib.load().turdb_cuda_last_error()


@pytest.fixture
def unbacked(monkeypatch):
    """Index objects whose every library call fails the test: validation has to happen first."""
    def no_library():
        raise AssertionError("the library was called")
    monkeypatch.setattr(_lib, "load", no_library)
    return [CudaHnswIndex(None, 8, 0, DistanceFunction.L2, 0) for _ in range(3)]


@pytest.mark.parametrize("op", [2, 3, -1])
def test_wrapper_rejects_unsupported_sort_operators(unbacked, op):
    with pytest.raises(ValueError):
        ShardedVectorScanBatch(unbacked, op, 10)


def test_wrapper_rejects_an_unknown_projection(unbacked):
    with pytest.raises(ValueError):
        ShardedVectorScanBatch(unbacked, VectorOp.L2Distance, 10, project=3)


@pytest.mark.parametrize("limit,offset", [(-1, 0), (10, -1), (2**32, 0), (513, 0), (500, 13), (0, 513)])
def test_wrapper_rejects_bad_windows(unbacked, limit, offset):
    with pytest.raises(ValueError):
        ShardedVectorScanBatch(unbacked, VectorOp.L2Distance, limit, offset)


def test_wrapper_accepts_the_largest_window(unbacked):
    op = ShardedVectorScanBatch(unbacked, VectorOp.CosineDistance, 500, 12, project=VectorOp.InnerProduct)
    assert (op.op, op.limit, op.offset, op.project, op.dim) == (1, 500, 12, 2, 8)


def test_wrapper_rejects_bad_shard_lists(unbacked):
    with pytest.raises(ValueError):
        ShardedVectorScanBatch([], VectorOp.L2Distance, 10)
    with pytest.raises(ValueError):
        ShardedVectorScanBatch(unbacked * 11, VectorOp.L2Distance, 10)  # 33 shards
    with pytest.raises(ValueError):  # dimension mismatch between shards
        ShardedVectorScanBatch(unbacked + [CudaHnswIndex(None, 7, 0, DistanceFunction.L2, 0)], VectorOp.L2Distance, 10)


@pytest.mark.parametrize("literals", [
    np.zeros((3, 7), np.float32),      # wrong dimension
    np.zeros((3, 8), np.int32),        # not floating point
    np.zeros((3, 8), object),
    np.zeros((2, 3, 8), np.float32),   # not [nq, dim]
])
def test_wrapper_rejects_bad_literals_before_the_library(unbacked, literals):
    with pytest.raises(ValueError):
        ShardedVectorScanBatch(unbacked, VectorOp.CosineDistance, 10).execute(literals)
