"""Builds tests/user_functor/my_hessians.cu OUT OF TREE (a temporary directory, the user's own nvcc command line) and loads it:
scalar objectives with analytic Hessians register their launch tables and Hessian launchers at load time. Also: the host side of the
analytic Hessian (the same __host__ __device__ partial2() the kernels compile)."""
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
MYH_F_QUADFORM, MYH_F_STYBLINSKI = 1301, 1302

_lib = None


def build_and_load():
    """compile once per process; returns the ctypes handle of the user's library"""
    global _lib
    if _lib is not None:
        return _lib
    from parallelnonlinearoptimizationlibrary_b200 import capi, hostapi
    capi.load_library()
    hostapi.lib()
    d = tempfile.mkdtemp(prefix="pnol_user_hessian_")
    out = os.path.join(d, "libmy_hessians.so")
    cmd = [user_functor_lib.nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-fmad=false", "-Xcompiler",
           "-fPIC,-ffp-contract=off", "-I" + os.path.join(ROOT, "include"), "-I" + SRC, "-shared", "-o", out,
           os.path.join(SRC, "my_hessians.cu"), "-L" + LIBDIR, "-lpnol_b200", "-lpnol_b200_host", "-Xlinker", "-rpath", "-Xlinker", LIBDIR]
    subprocess.run(cmd, check=True, cwd=d, capture_output=True, text=True)
    _lib = C.CDLL(out, mode=C.RTLD_GLOBAL)
    return _lib


def _call(kind, x, scalars, ints, columns, ii, jj, npairs, out):
    u = build_and_load()
    columns = [np.ascontiguousarray(c, dtype=np.float64) for c in columns]
    P = user_jacobian_lib.params(scalars, columns)
    for i, v in enumerate(ints):
        P.ints[i] = int(v)
    x = np.ascontiguousarray(x, dtype=np.float64)
    p = lambda a: None if a is None else C.c_void_p(a.ctypes.data)       # noqa: E731
    st = u.my_host_partial2(int(kind), C.byref(P), p(x), int(x.size), p(ii), p(jj), C.c_longlong(npairs), p(out))
    assert st == 0, kind
    return out


def host_hessian(kind, x, scalars=(), ints=(), columns=()):
    """the n x n matrix of the functor's partial2() run on the host, upper triangle computed and mirrored"""
    n = int(np.size(x))
    return _call(kind, x, scalars, ints, columns, None, None, 0, np.empty((n, n)))


def host_partial2(kind, x, ii, jj, scalars=(), ints=(), columns=()):
    """d2f / dx_ii[k] dx_jj[k] of the functor's partial2() run on the host (ii[k] <= jj[k])"""
    ii, jj = np.ascontiguousarray(ii, dtype=np.int32), np.ascontiguousarray(jj, dtype=np.int32)
    assert ii.size == jj.size and np.all(ii <= jj)
    return _call(kind, x, scalars, ints, columns, ii, jj, ii.size, np.empty(ii.size))
