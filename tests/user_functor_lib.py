"""Builds tests/user_functor/my_objectives.cu OUT OF TREE (a temporary directory, the user's own nvcc command line) and loads it:
objectives that are not built into libpnol_b200.so register their launch tables at load time (include/pnol_b200.h:
pnol_register_functor; include/pnol/device/functor_kernels.cuh)."""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "user_functor")
LIBDIR = os.path.join(ROOT, "parallelnonlinearoptimizationlibrary_b200", "lib")
MY_F_TRID, MY_F_STYBLINSKI, MY_F_GAUSSFIT = 1001, 1002, 2001

_lib = None


def nvcc():
    return shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"


def build_user_library(source, with_host_lib=True):
    """compiles tests/user_functor/<source> OUT OF TREE (a temporary directory, the user's own nvcc command line) into its own
    lib<name>.so, linked against libpnol_b200.so and, with_host_lib, libpnol_b200_host.so, and loads it RTLD_GLOBAL: the kinds it
    defines register with the library at load time"""
    from parallelnonlinearoptimizationlibrary_b200 import capi, hostapi
    capi.load_library()
    hostapi.lib()
    name = os.path.splitext(source)[0]
    d = tempfile.mkdtemp(prefix="pnol_%s_" % name)
    out = os.path.join(d, "lib%s.so" % name)
    cmd = [nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-fmad=false", "-Xcompiler", "-fPIC,-ffp-contract=off",
           "-I" + os.path.join(ROOT, "include"), "-I" + SRC, "-shared", "-o", out, os.path.join(SRC, source),
           "-L" + LIBDIR, "-lpnol_b200"] + (["-lpnol_b200_host"] if with_host_lib else []) + ["-Xlinker", "-rpath", "-Xlinker", LIBDIR]
    subprocess.run(cmd, check=True, cwd=d, capture_output=True, text=True)
    return C.CDLL(out, mode=C.RTLD_GLOBAL)


def build_and_load():
    """compile once per process; returns the ctypes handle of the user's library"""
    global _lib
    if _lib is None:
        _lib = build_user_library("my_objectives.cu")
        _lib.my_host_eval.restype = C.c_double
    return _lib
