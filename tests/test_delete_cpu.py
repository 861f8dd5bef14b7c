"""turdb_cuda_index_delete without a device: the C entry's argument checks and the Python wrapper's validation, which
must reject bad input before the library is called."""
import ctypes as C

import numpy as np
import pytest

from turdb_b200 import _lib
from turdb_b200.hnsw import CudaHnswIndex, DistanceFunction


def test_delete_null_index_is_an_invalid_argument():
    L = _lib.load()
    ids = np.zeros(1, np.uint32)
    out = C.c_uint64(7)
    rc = L.turdb_cuda_index_delete(None, 1, ids.ctypes.data_as(C.POINTER(C.c_uint32)), C.byref(out))
    assert rc == _lib.ERR_INVALID_ARGUMENT
    assert b"idx is null" in L.turdb_cuda_last_error()
    assert out.value == 7  # nothing written on failure
    assert L.turdb_cuda_index_delete(None, 0, None, None) == _lib.ERR_INVALID_ARGUMENT


def test_delete_null_ids_with_rows_is_an_invalid_argument():
    L = _lib.load()
    assert L.turdb_cuda_index_delete(None, 3, None, None) == _lib.ERR_INVALID_ARGUMENT
    assert b"node_ids is null" in L.turdb_cuda_last_error()


@pytest.fixture
def unbacked(monkeypatch):
    """An index object of 5 nodes whose every library call fails the test: validation has to happen first."""
    def no_library():
        raise AssertionError("the library was called")
    monkeypatch.setattr(_lib, "load", no_library)
    return CudaHnswIndex(None, 8, 5, DistanceFunction.L2, 0)


@pytest.mark.parametrize("ids", [
    np.array([5], np.uint32),             # id == n
    np.array([0, 7], np.int64),           # id > n
    np.array([-1], np.int64),             # negative
    np.array([2 ** 32], np.uint64),       # beyond u32 (would wrap)
    np.array([1.0, 2.0]),                 # not integers
    np.array([True, False]),
    np.array([[0, 1]], np.uint32),        # not [n]
    np.uint32(1),                         # a scalar
    np.array(["1"]),
])
def test_wrapper_rejects_bad_ids_before_the_library(unbacked, ids):
    with pytest.raises(ValueError):
        unbacked.delete(ids)


def test_wrapper_passes_valid_ids_as_u32(monkeypatch):
    seen = {}

    class Fake:
        def turdb_cuda_index_delete(self, h, n, ptr, out):
            seen["n"] = n
            seen["ids"] = None if ptr is None else np.ctypeslib.as_array(ptr, shape=(n,)).copy()
            out._obj.value = 3
            return _lib.OK

    monkeypatch.setattr(_lib, "load", lambda: Fake())
    idx = CudaHnswIndex(None, 8, 5, DistanceFunction.L2, 0)
    assert idx.delete(np.array([4, 0, 4], np.int64)) == 3
    assert seen["n"] == 3 and seen["ids"].tolist() == [4, 0, 4]
    assert idx.delete([]) == 3 and seen["n"] == 0 and seen["ids"] is None
    assert idx.n == 5  # node ids stay as they are
