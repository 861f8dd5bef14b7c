"""turdb_cuda_sql_range_batch without a device: the C entries' argument checks and the Python wrapper's validation, which
must reject bad input before the library is called."""
import ctypes as C

import numpy as np
import pytest

from turdb_b200 import _lib
from turdb_b200.hnsw import CudaHnswIndex, DistanceFunction
from turdb_b200.sql_operator import RangeCmp, VectorOp, VectorRangeScanBatch, range_direction_supported


def test_null_index_is_an_invalid_argument():
    L = _lib.load()
    q = np.zeros((1, 8), np.float32)
    r = np.ones(1)
    rows = np.zeros(4, np.uint64)
    cnt = np.zeros(1, np.uint32)
    rc = L.turdb_cuda_sql_range_batch(None, q.ctypes.data_as(C.POINTER(C.c_float)), 8, 1, 0, 0,
                                      r.ctypes.data_as(C.POINTER(C.c_double)), 4, 0,
                                      rows.ctypes.data_as(C.POINTER(C.c_uint64)), None, cnt.ctypes.data_as(C.POINTER(C.c_uint32)))
    assert rc == _lib.ERR_INVALID_ARGUMENT
    assert b"null" in L.turdb_cuda_last_error()
    assert L.turdb_cuda_sql_range_batch_device(None, None, 8, 1, 0, 0, None, 4, 0, None, None, None, None) == _lib.ERR_INVALID_ARGUMENT


def test_near_direction_only():
    supported = {(o, c) for o in VectorOp for c in RangeCmp if range_direction_supported(o, c)}
    assert supported == {(VectorOp.L2Distance, RangeCmp.Lt), (VectorOp.L2Distance, RangeCmp.Le),
                         (VectorOp.CosineDistance, RangeCmp.Lt), (VectorOp.CosineDistance, RangeCmp.Le),
                         (VectorOp.InnerProduct, RangeCmp.Gt), (VectorOp.InnerProduct, RangeCmp.Ge)}


@pytest.fixture
def unbacked(monkeypatch):
    """An index object whose every library call fails the test: validation has to happen first."""
    def no_library():
        raise AssertionError("the library was called")
    monkeypatch.setattr(_lib, "load", no_library)
    return CudaHnswIndex(None, 8, 0, DistanceFunction.L2, 0)


@pytest.mark.parametrize("op,cmp", [(0, 2), (0, 3), (1, 2), (1, 3), (2, 0), (2, 1), (3, 0), (0, 4), (-1, 0)])
def test_wrapper_rejects_unsupported_operators(unbacked, op, cmp):
    with pytest.raises(ValueError):
        VectorRangeScanBatch(unbacked, op, cmp, 10)


@pytest.mark.parametrize("limit,offset", [(-1, 0), (10, -1), (2**32, 0)])
def test_wrapper_rejects_bad_windows(unbacked, limit, offset):
    with pytest.raises(ValueError):
        VectorRangeScanBatch(unbacked, VectorOp.L2Distance, RangeCmp.Lt, limit, offset)


Q = np.zeros((3, 8), np.float32)
R = np.ones(3)


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
        VectorRangeScanBatch(unbacked, VectorOp.CosineDistance, RangeCmp.Le, 10).execute(literals, radius)
