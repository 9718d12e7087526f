"""Builds tests/user_functor/my_wide_models.cu OUT OF TREE (a temporary directory, the user's own nvcc command line) and loads it:
a residual model of any width n whose launch table registers at load time. Also its host side (the same __host__ __device__
definitions the kernels compile) and a numpy restatement of its analytic Jacobian."""
import ctypes as C

import numpy as np

import user_functor_lib
import user_jacobian_lib

MYW_F_WIDE = 2201

_lib = None


def build_and_load():
    """compile once per process; returns the ctypes handle of the user's library"""
    global _lib
    if _lib is None:
        _lib = user_functor_lib.build_user_library("my_wide_models.cu")
    return _lib


def columns(m, rng, tiny_rows=(), bare_rows=()):
    """(t, s, y) of m rows; rows in tiny_rows get t = 2^-760 and s = y = 0, so that their forward differences are below 2^-700;
    rows in bare_rows get s = y = 0, so that r_i = -(x_a t_i) keeps the difference of a tiny x_a and a tinier step"""
    t = rng.uniform(0.5, 2.0, m)
    s = rng.uniform(-1.5, 1.5, m)
    y = rng.normal(size=m)
    bare = np.asarray(bare_rows, dtype=np.int64)
    s[bare], y[bare] = 0.0, 0.0
    tiny = np.asarray(tiny_rows, dtype=np.int64)
    t[tiny], s[tiny], y[tiny] = 2.0 ** -760, 0.0, 0.0
    return t, s, y


def cols_ab(m, n):
    i = np.arange(m, dtype=np.int64)
    return i % n, (7 * i + 3) % n


def _p(a):
    return C.c_void_p(a.ctypes.data)


def host_rows(cols, x, want_j=True, i0=0, i1=None):
    """(J, F) of rows [i0, i1) (default: all) of the model's jacobian() / residual() run on the host"""
    u = build_and_load()
    cols = [np.ascontiguousarray(c, dtype=np.float64) for c in cols]
    P = user_jacobian_lib.params((), cols)
    x = np.ascontiguousarray(x, dtype=np.float64)
    i1 = P.m if i1 is None else i1
    n = x.size
    J = np.empty((i1 - i0, n)) if want_j else None
    F = np.empty(i1 - i0)
    u.my_wide_host_rows(C.byref(P), _p(x), int(n), C.c_longlong(i0), C.c_longlong(i1), _p(J) if want_j else None, _p(F))
    return J, F


def host_fd_jacobian(cols, x, dx):
    """(J, F): the host's stencil residuals with numpy's IEEE quotient (r_j - r_0) / dx_j"""
    u = build_and_load()
    cols = [np.ascontiguousarray(c, dtype=np.float64) for c in cols]
    P = user_jacobian_lib.params((), cols)
    x, dx = np.ascontiguousarray(x, dtype=np.float64), np.ascontiguousarray(dx, dtype=np.float64)
    m, n = P.m, x.size
    Rp = np.empty((m, n))
    u.my_wide_host_stencils(C.byref(P), _p(x), _p(dx), int(n), C.c_longlong(m), _p(Rp))
    _, F = host_rows(cols, x, want_j=False)
    with np.errstate(all="ignore"):
        return (Rp - F[:, None]) / dx[None, :], F


def np_jacobian(cols, x):
    """jacobian() restated in numpy, in its operation order"""
    t, s, _ = cols
    m, n = t.size, x.size
    a, b = cols_ab(m, n)
    xb = x[b]
    ja, jb = -t, -((xb + xb) * s)
    J = np.zeros((m, n))
    rows = np.arange(m)
    same = a == b
    J[rows[~same], a[~same]] = ja[~same]
    J[rows[~same], b[~same]] = jb[~same]
    J[rows[same], a[same]] = ja[same] + jb[same]
    return J
