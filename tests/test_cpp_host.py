"""The C++17 host mirror (include/turdb_cuda.hpp) — the native-language host side over the C ABI (the reference is
compiled code; its Rust toolchain is absent here).  Compiled with g++ against the in-tree library."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIBDIR = os.path.join(ROOT, "turdb_b200")


@pytest.fixture(scope="module")
def host_mirror_exe(tmp_path_factory):
    """The mirror's test program, compiled into a temporary directory: the source tree may be read-only."""
    from turdb_b200 import build as tb
    tb.build_library()
    src = os.path.join(ROOT, "tests", "cpp", "host_mirror_test.cpp")
    exe = str(tmp_path_factory.mktemp("cpp") / "host_mirror_test.bin")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"), src, "-o", exe,
                           "-L", LIBDIR, "-lturdb_cuda", f"-Wl,-rpath,{LIBDIR}"])
    return exe


def test_cpp_mirror_compiles_and_fails_loudly_without_a_device(host_mirror_exe):
    import ctypes
    from turdb_b200 import _lib
    c = ctypes.c_int32(0)
    if _lib.load().turdb_cuda_device_count(ctypes.byref(c)) == 0 and c.value > 0:
        pytest.skip("a device is present: the full run below covers it")
    out = subprocess.run([host_mirror_exe, "--no-device"], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr
    assert "no-device checks ok" in out.stdout


@pytest.mark.gpu
def test_cpp_mirror_end_to_end(gpu_required, host_mirror_exe):
    out = subprocess.run([host_mirror_exe], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr + out.stdout
    assert "all checks ok" in out.stdout
