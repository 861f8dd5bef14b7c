"""CPU restatement of turdb_cuda_index_compact on flat graph arrays (the turdb_cuda_graph layout that export_graph and
OracleGraph.export produce).  Test infrastructure: the per-row part of the rule is here, the list repair is
tests/cpp/compact_reference.cpp, compiled on first use into a temporary directory (the source tree may be read-only)."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
INVALID = 0xFFFFFFFF
_lib = None


def _load():
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="turdb_compact_ref_"), "libcompact_reference.so")
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-mavx2", "-mfma", "-ffp-contract=off", "-fPIC", "-shared",
                               "-Wall", "-o", out, os.path.join(HERE, "cpp", "compact_reference.cpp")])
        _lib = C.CDLL(out)
        _lib.tcr_compact_lists.restype = None
        _lib.tcr_compact_lists.argtypes = [C.c_uint32, C.c_uint64] + [C.c_void_p] * 14
    return _lib


def compact(arrays: dict, live) -> tuple[dict, np.ndarray]:
    """(compacted arrays, old -> new map) for the graph `arrays` with the nodes whose `live` entry is False removed."""
    live = np.asarray(live, bool)
    n = live.shape[0]
    o2n = np.where(live, np.cumsum(live) - 1, INVALID).astype(np.uint32)
    if live.all():
        return {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in arrays.items()}, o2n
    a = {k: (np.ascontiguousarray(v) if isinstance(v, np.ndarray) else v) for k, v in arrays.items()}
    levels = a["levels"][live]
    up_base = np.where(levels > 0, np.cumsum(levels.astype(np.uint64)) - levels, INVALID).astype(np.uint32)
    slots = int(levels.astype(np.uint64).sum())
    n_live = int(live.sum())
    out = dict(vectors=np.ascontiguousarray(a["vectors"][live]), row_ids=a["row_ids"][live].copy(), levels=levels,
               l0_adj=np.full((n_live, 32), INVALID, np.uint32), l0_cnt=np.zeros(n_live, np.uint8), up_base=up_base,
               up_adj=np.full((slots, 16), INVALID, np.uint32), up_cnt=np.zeros(slots, np.uint8))
    if n_live:
        p = lambda x: x.ctypes.data if x.size else None  # noqa: E731
        live8 = live.astype(np.uint8)
        _load().tcr_compact_lists(a["vectors"].shape[1], n, p(a["vectors"]), p(a["levels"]), p(a["l0_adj"]),
                                  p(a["l0_cnt"]), p(a["up_base"]), p(a["up_adj"]), p(a["up_cnt"]), p(live8), p(o2n),
                                  p(up_base), p(out["l0_adj"]), p(out["l0_cnt"]), p(out["up_adj"]), p(out["up_cnt"]))
    entry, max_level = int(arrays["entry"]), int(arrays["max_level"])
    if n_live == 0:
        entry, max_level = INVALID, 0
    elif entry != INVALID and not live[entry]:  # the live node of the highest level, lowest new id among ties
        entry = int(np.argmax(levels))
        max_level = int(levels[entry])
    elif entry != INVALID:
        entry = int(o2n[entry])
    out["entry"], out["max_level"] = entry, max_level
    return out, o2n
