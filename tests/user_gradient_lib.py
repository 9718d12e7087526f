"""Builds tests/user_functor/my_gradients.cu OUT OF TREE (a temporary directory, the user's own nvcc command line) and loads it:
scalar objectives with analytic gradients register their launch tables and gradient launchers at load time. Also: the host side of
the analytic gradient (the same __host__ __device__ partial() the kernels compile) and of the shared host/device math."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

import user_functor_lib
import user_jacobian_lib

ROOT = user_functor_lib.ROOT
SRC = user_functor_lib.SRC
LIBDIR = user_functor_lib.LIBDIR
MYG_F_TRID, MYG_F_STYBLINSKI = 1201, 1202

_lib = None


def build_and_load():
    """compile once per process; returns the ctypes handle of the user's library"""
    global _lib
    if _lib is not None:
        return _lib
    from parallelnonlinearoptimizationlibrary_b200 import capi, hostapi
    capi.load_library()
    hostapi.lib()
    d = tempfile.mkdtemp(prefix="pnol_user_gradient_")
    out = os.path.join(d, "libmy_gradients.so")
    cmd = [user_functor_lib.nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-fmad=false", "-Xcompiler",
           "-fPIC,-ffp-contract=off", "-I" + os.path.join(ROOT, "include"), "-I" + SRC, "-shared", "-o", out,
           os.path.join(SRC, "my_gradients.cu"), "-L" + LIBDIR, "-lpnol_b200", "-lpnol_b200_host", "-Xlinker", "-rpath", "-Xlinker", LIBDIR]
    subprocess.run(cmd, check=True, cwd=d, capture_output=True, text=True)
    _lib = C.CDLL(out, mode=C.RTLD_GLOBAL)
    return _lib


def host_partials(kind, x, scalars=(), ints=(), columns=(), idx=None):
    """df/dx_j of the functor's partial() run on the host, for j in idx (default: every coordinate)"""
    u = build_and_load()
    columns = [np.ascontiguousarray(c, dtype=np.float64) for c in columns]
    P = user_jacobian_lib.params(scalars, columns)
    for i, v in enumerate(ints):
        P.ints[i] = int(v)
    x = np.ascontiguousarray(x, dtype=np.float64)
    idx = np.arange(x.size, dtype=np.int32) if idx is None else np.ascontiguousarray(idx, dtype=np.int32)
    g = np.empty(idx.size)
    st = u.my_host_partials(int(kind), C.byref(P), C.c_void_p(x.ctypes.data), int(x.size), C.c_void_p(idx.ctypes.data), int(idx.size),
                            C.c_void_p(g.ctypes.data))
    assert st == 0, kind
    return g


def host_math(which, x):
    """pnol_math.h on the host: which = "sin2pi" | "cos2pi" | "exp" """
    u = build_and_load()
    x = np.ascontiguousarray(x, dtype=np.float64)
    out = np.empty_like(x)
    assert u.my_host_math({"sin2pi": 0, "cos2pi": 1, "exp": 2}[which], C.c_void_p(x.ctypes.data), C.c_longlong(x.size),
                          C.c_void_p(out.ctypes.data)) == 0
    return out
