"""Builds tests/user_functor/my_jacobians.cu OUT OF TREE (a temporary directory, the user's own nvcc command line) and loads it:
residual models with analytic Jacobians register their launch tables at load time. Also: the host side of the analytic Jacobian
(the same __host__ __device__ definitions the kernels compile) and a ctypes mirror of pnol_functor_params."""
import ctypes as C

import numpy as np

import user_functor_lib

MYJ_F_LORENTZ, MYJ_F_GAUSS, MYJ_F_GAUSS_V1, MYJ_F_GAUSS_NOJAC = 2101, 2102, 2103, 2104

_lib = None


class FunctorParams(C.Structure):
    """pnol_functor_params (include/pnol_b200.h)"""
    _fields_ = [("scalars", C.c_double * 8), ("ints", C.c_longlong * 4), ("col", C.c_void_p * 8), ("m", C.c_longlong)]


def build_and_load():
    """compile once per process; returns the ctypes handle of the user's library"""
    global _lib
    if _lib is None:
        _lib = user_functor_lib.build_user_library("my_jacobians.cu")
    return _lib


def params(scalars=(), columns=()):
    """host-side pnol_functor_params over numpy columns (kept alive by the caller)"""
    P = FunctorParams()
    for i, v in enumerate(scalars):
        P.scalars[i] = float(v)
    for i, c in enumerate(columns):
        assert c.dtype == np.float64 and c.flags["C_CONTIGUOUS"]
        P.col[i] = c.ctypes.data
    P.m = int(columns[0].size) if columns else 0
    return P


def host_jacobian(kind, scalars, columns, x, rows=None):
    """(J[rows], F[rows]) of the functor's jacobian() / residual() run on the host"""
    u = build_and_load()
    columns = [np.ascontiguousarray(c, dtype=np.float64) for c in columns]
    P = params(scalars, columns)
    x = np.ascontiguousarray(x, dtype=np.float64)
    rows = np.arange(P.m, dtype=np.int64) if rows is None else np.ascontiguousarray(rows, dtype=np.int64)
    J = np.empty((rows.size, x.size))
    F = np.empty(rows.size)
    st = u.my_host_jacobian_rows(int(kind), C.byref(P), C.c_void_p(x.ctypes.data), int(x.size), C.c_void_p(rows.ctypes.data),
                                 C.c_longlong(rows.size), C.c_void_p(J.ctypes.data), C.c_void_p(F.ctypes.data))
    assert st == 0, kind
    return J, F
