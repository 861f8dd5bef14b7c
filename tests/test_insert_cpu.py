"""turdb_cuda_index_insert without a device: the C entry's argument checks and the Python wrapper's validation, which
must reject bad input before the library is called."""
import ctypes as C

import numpy as np
import pytest

from turdb_b200 import _lib
from turdb_b200.hnsw import CudaHnswIndex, DistanceFunction


def test_insert_null_index_is_an_invalid_argument():
    L = _lib.load()
    bp = _lib.BuildParams(8, 16, 100, 1, 1, 0)
    x = np.zeros((1, 8), np.float32)
    rid = np.zeros(1, np.uint64)
    rnd = np.ones(1, np.float64)
    rc = L.turdb_cuda_index_insert(None, C.byref(bp), 1, x.ctypes.data_as(C.POINTER(C.c_float)),
                                   rid.ctypes.data_as(C.POINTER(C.c_uint64)), rnd.ctypes.data_as(C.POINTER(C.c_double)))
    assert rc == _lib.ERR_INVALID_ARGUMENT
    assert b"null" in L.turdb_cuda_last_error()


@pytest.fixture
def unbacked(monkeypatch):
    """An index object whose every library call fails the test: validation has to happen first."""
    def no_library():
        raise AssertionError("the library was called")
    monkeypatch.setattr(_lib, "load", no_library)
    return CudaHnswIndex(None, 8, 0, DistanceFunction.L2, 0, build_params=(16, 100, 1))


GOOD = dict(vectors=np.zeros((3, 8), np.float32), row_ids=np.arange(3, dtype=np.uint64), random_values=np.ones(3))


@pytest.mark.parametrize("field,value", [
    ("vectors", np.zeros((3, 7), np.float32)),          # wrong dimension
    ("vectors", np.zeros(8, np.float32)),               # not [n, dim]
    ("vectors", np.zeros((3, 8), np.int32)),            # not floating point
    ("vectors", np.zeros((3, 8), object)),
    ("row_ids", np.arange(2, dtype=np.uint64)),         # one per row
    ("row_ids", np.arange(3, dtype=np.float64)),        # not integers
    ("row_ids", np.array([0, -1, 2], np.int64)),
    ("random_values", np.ones(4)),
    ("random_values", np.ones(3, np.int64)),
    ("random_values", None),
    ("row_ids", None),
])
def test_wrapper_rejects_bad_input_before_the_library(unbacked, field, value):
    args = dict(GOOD)
    args[field] = value
    with pytest.raises(ValueError):
        unbacked.insert(**args)
    assert unbacked.n == 0


def test_wrapper_needs_parameters_without_a_build(monkeypatch):
    monkeypatch.setattr(_lib, "load", lambda: (_ for _ in ()).throw(AssertionError("the library was called")))
    idx = CudaHnswIndex(None, 8, 0, DistanceFunction.L2, 0)  # as from_graph leaves it
    with pytest.raises(ValueError, match="required"):
        idx.insert(**GOOD)
    with pytest.raises(ValueError, match="required"):
        idx.insert(**GOOD, m=16, ef_construction=100)
