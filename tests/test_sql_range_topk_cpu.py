"""turdb_cuda_sql_range_topk_batch without a device: the C entries' argument checks (operators and window are checked
before the index) and the Python wrapper's validation, which must reject bad input before the library is called."""
import ctypes as C

import numpy as np
import pytest

from turdb_b200 import _lib
from turdb_b200.hnsw import CudaHnswIndex, DistanceFunction
from turdb_b200.sql_operator import RangeCmp, VectorOp, VectorRangeTopKBatch

Q = np.zeros((3, 8), np.float32)
R = np.ones(3)


def host_entry(where_op, cmp, order_op, limit, offset, proj_op=0, project=False):
    L = _lib.load()
    size = 3 * min(max(limit, 1), 512)  # a rejected window is never written
    rows = np.zeros(size, np.uint64)
    keys = np.zeros(size)
    proj = np.zeros(size)
    cnt = np.zeros(3, np.uint32)
    d = C.POINTER(C.c_double)
    return L.turdb_cuda_sql_range_topk_batch(None, Q.ctypes.data_as(C.POINTER(C.c_float)), 8, 3, where_op, cmp,
                                             R.ctypes.data_as(d), order_op, proj_op, limit, offset,
                                             rows.ctypes.data_as(C.POINTER(C.c_uint64)), keys.ctypes.data_as(d),
                                             proj.ctypes.data_as(d) if project else None,
                                             cnt.ctypes.data_as(C.POINTER(C.c_uint32)))


def device_entry(where_op, cmp, order_op, limit, offset):
    return _lib.load().turdb_cuda_sql_range_topk_batch_device(None, None, 8, 3, where_op, cmp, None, order_op, 0, limit,
                                                              offset, None, None, None, None, None)


def test_null_index_is_an_invalid_argument():
    L = _lib.load()
    assert host_entry(1, 0, 1, 10, 0) == _lib.ERR_INVALID_ARGUMENT
    assert b"null" in L.turdb_cuda_last_error()
    assert device_entry(1, 0, 1, 10, 0) == _lib.ERR_INVALID_ARGUMENT
    assert b"null" in L.turdb_cuda_last_error()


@pytest.mark.parametrize("entry", [host_entry, device_entry])
@pytest.mark.parametrize("where_op,cmp", [(0, 2), (0, 3), (1, 2), (1, 3), (2, 0), (2, 1)])
def test_far_direction_is_unsupported(entry, where_op, cmp):
    assert entry(where_op, cmp, 0, 10, 0) == _lib.ERR_UNSUPPORTED
    assert b"near direction" in _lib.load().turdb_cuda_last_error()


@pytest.mark.parametrize("entry", [host_entry, device_entry])
def test_order_by_inner_product_is_unsupported(entry):
    assert entry(2, 2, 2, 10, 0) == _lib.ERR_UNSUPPORTED
    assert b"<#>" in _lib.load().turdb_cuda_last_error()


@pytest.mark.parametrize("entry", [host_entry, device_entry])
@pytest.mark.parametrize("limit,offset", [(513, 0), (0, 513), (500, 13), (2**32 - 1, 1)])
def test_window_past_the_heap_limit_is_unsupported(entry, limit, offset):
    assert entry(1, 1, 1, limit, offset) == _lib.ERR_UNSUPPORTED
    assert b"limit + offset" in _lib.load().turdb_cuda_last_error()


def test_unknown_operators_are_invalid_arguments():
    assert host_entry(3, 0, 0, 10, 0) == _lib.ERR_INVALID_ARGUMENT
    assert host_entry(0, 4, 0, 10, 0) == _lib.ERR_INVALID_ARGUMENT
    assert host_entry(0, 0, 0, 10, 0, proj_op=3, project=True) == _lib.ERR_INVALID_ARGUMENT
    assert host_entry(0, 0, 0, 500, 12) == _lib.ERR_INVALID_ARGUMENT  # limit + offset = 512 passes: the index is null


@pytest.fixture
def unbacked(monkeypatch):
    """An index object whose every library call fails the test: validation has to happen first."""
    def no_library():
        raise AssertionError("the library was called")
    monkeypatch.setattr(_lib, "load", no_library)
    return CudaHnswIndex(None, 8, 0, DistanceFunction.L2, 0)


@pytest.mark.parametrize("where_op,cmp,order_op", [
    (0, 2, 0), (0, 3, 0), (1, 2, 1), (1, 3, 1), (2, 0, 0), (2, 1, 1),  # far direction
    (3, 0, 0), (0, 4, 0), (-1, 0, 0),                                  # unknown WHERE operator / comparison
    (0, 0, 2), (2, 2, 2),                                              # ORDER BY <#>
    (0, 0, 3), (0, 0, -1),                                             # unknown ORDER BY operator
])
def test_wrapper_rejects_unsupported_operators(unbacked, where_op, cmp, order_op):
    with pytest.raises(ValueError):
        VectorRangeTopKBatch(unbacked, where_op, cmp, order_op, 10)


def test_wrapper_rejects_an_unknown_projection(unbacked):
    with pytest.raises(ValueError):
        VectorRangeTopKBatch(unbacked, VectorOp.L2Distance, RangeCmp.Lt, VectorOp.L2Distance, 10, project=3)


@pytest.mark.parametrize("limit,offset", [(-1, 0), (10, -1), (2**32, 0), (513, 0), (500, 13), (0, 513)])
def test_wrapper_rejects_bad_windows(unbacked, limit, offset):
    with pytest.raises(ValueError):
        VectorRangeTopKBatch(unbacked, VectorOp.L2Distance, RangeCmp.Lt, VectorOp.L2Distance, limit, offset)


def test_wrapper_accepts_the_largest_window(unbacked):
    op = VectorRangeTopKBatch(unbacked, VectorOp.InnerProduct, RangeCmp.Ge, VectorOp.CosineDistance, 500, 12,
                              project=VectorOp.InnerProduct)
    assert (op.where_op, op.cmp, op.order_op, op.limit, op.offset) == (2, 3, 1, 500, 12)


@pytest.mark.parametrize("literals,radius", [
    (np.zeros((3, 7), np.float32), R),           # wrong dimension
    (np.zeros((3, 8), np.int32), R),             # literals not floating point
    (np.zeros((3, 8), object), R),
    (np.zeros((2, 3, 8), np.float32), R),        # not [nq, dim]
    (Q, np.ones(2)),                             # one radius per statement
    (Q, np.ones(4)),
    (Q, np.ones((3, 1))),
    (Q, np.array(["a", "b", "c"])),              # radius not a number
    (Q, None),
])
def test_wrapper_rejects_bad_input_before_the_library(unbacked, literals, radius):
    with pytest.raises(ValueError):
        VectorRangeTopKBatch(unbacked, VectorOp.CosineDistance, RangeCmp.Le, VectorOp.CosineDistance, 10).execute(literals,
                                                                                                                   radius)
