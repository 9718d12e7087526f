"""Builds tests/user_functor/my_simplex_objectives.cu OUT OF TREE (a temporary directory, the user's own nvcc command line) the way
tests/user_functor_lib.py builds my_objectives.cu, and loads it: the four simplex test objectives register their launch tables, and with
them their batched simplex launchers, at load time."""
import ctypes as C
import os
import subprocess
import tempfile

from user_functor_lib import LIBDIR, ROOT, SRC, nvcc

MYS_F_NEGATIVE, MYS_F_QUANTIZED, MYS_F_SIGNED_ZERO, MYS_F_NAN_REGION = 1401, 1402, 1403, 1404
NAMES = {MYS_F_NEGATIVE: "negative", MYS_F_QUANTIZED: "quantized", MYS_F_SIGNED_ZERO: "signed_zero", MYS_F_NAN_REGION: "nan_region"}

_lib = None


def build_and_load():
    """compile once per process; returns the ctypes handle of the user's library"""
    global _lib
    if _lib is not None:
        return _lib
    from parallelnonlinearoptimizationlibrary_b200 import capi, hostapi
    capi.load_library()
    hostapi.lib()
    d = tempfile.mkdtemp(prefix="pnol_user_simplex_")
    out = os.path.join(d, "libmy_simplex_objectives.so")
    cmd = [nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-fmad=false", "-Xcompiler", "-fPIC,-ffp-contract=off",
           "-I" + os.path.join(ROOT, "include"), "-I" + SRC, "-shared", "-o", out, os.path.join(SRC, "my_simplex_objectives.cu"),
           "-L" + LIBDIR, "-lpnol_b200", "-Xlinker", "-rpath", "-Xlinker", LIBDIR]
    subprocess.run(cmd, check=True, cwd=d, capture_output=True, text=True)
    _lib = C.CDLL(out, mode=C.RTLD_GLOBAL)
    assert _lib.my_simplex_registration_status() == 0
    return _lib
