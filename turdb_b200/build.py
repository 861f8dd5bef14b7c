"""In-tree build of libturdb_cuda.so (nvcc, sm_100a only).  `python -m turdb_b200.build`."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libturdb_cuda.so")
# translation units: (source, extra -D switches, object name).  The traversal kernel's instantiations are split per
# metric and form so that they compile in parallel (one nvcc process each).
UNITS = [("turdb_cuda.cu", [], "turdb_cuda.o")]
for _m, _mn in ((0, "l2"), (1, "cosine"), (2, "ip")):
    UNITS.append(("search_kernels_staged.cu", [f"TURDB_TU_METRIC={_m}"], f"search_staged_{_mn}.o"))
    UNITS.append(("search_kernels_direct.cu", [f"TURDB_TU_METRIC={_m}"], f"search_direct_{_mn}.o"))
DEPS = ["turdb_cuda.cu", "common.cuh", "hnsw_search.cuh", "search_kernels.h", "search_kernels_staged.cu", "search_kernels_direct.cu",
        "exact_search.cuh", "exact_abi.inl", "gather_probe.cuh", "hnsw_file.inl", "sql_topk.inl", "sql_range.inl", "graph_insert.inl",
        os.path.join("..", "..", "include", "turdb_cuda.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-Wall"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libturdb_cuda.so cannot be built (there is no CPU fallback)")


def is_stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, d)) > t for d in DEPS)


def _compile_all(out: str, defines: list[str], verbose: bool = False) -> str:
    """nvcc -c every unit in parallel (objects under build/<tag>/), then link the shared library."""
    from concurrent.futures import ThreadPoolExecutor
    tag = os.path.basename(out).replace(".so", "")
    odir = os.path.join(HERE, "build", tag)
    os.makedirs(odir, exist_ok=True)
    nvcc = _nvcc()

    def one(unit):
        src, defs, obj = unit
        cmd = [nvcc, *NVCC_FLAGS, *[f"-D{d}" for d in defs + defines], "-c", "-o", os.path.join(odir, obj), os.path.join(CSRC, src)]
        if verbose:
            cmd[1:1] = ["-Xptxas", "-v"]
            print(" ".join(cmd), file=sys.stderr)
        r = subprocess.run(cmd, cwd=HERE, capture_output=True, text=True)
        return unit, r

    with ThreadPoolExecutor(max_workers=min(len(UNITS), os.cpu_count() or 2)) as ex:
        results = list(ex.map(one, UNITS))
    for unit, r in results:
        if verbose or r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {unit[0]} {unit[1]}")
    objs = [os.path.join(odir, u[2]) for u in UNITS]
    subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", out, *objs], cwd=HERE)
    return out


def build_library(force: bool = False, verbose: bool = False) -> str:
    if not force and not is_stale():
        return LIB
    return _compile_all(LIB, [], verbose)


def build_variant(name: str, defines: list[str]) -> str:
    """A/B builds for measurement (tools/sweep.py --libs): same sources, extra -D switches, loaded through the
    TURDB_CUDA_LIB override of _lib.py.  Written next to the library as libturdb_cuda.<name>.so."""
    return _compile_all(os.path.join(HERE, f"libturdb_cuda.{name}.so"), defines)


if __name__ == "__main__":
    for arg in sys.argv[1:]:
        if arg.startswith("--variant="):  # --variant=name:DEF1=1,DEF2=0
            vname, _, defs = arg[len("--variant="):].partition(":")
            print(build_variant(vname, [d for d in defs.split(",") if d]))
            sys.exit(0)
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
