"""Analytic Jacobians (PNOL_JAC_ANALYTIC) without a GPU: the host side of the one __host__ __device__ definition per model
(include/pnol/functors.hpp: R::jacobian, lorentz_term_grad) against a numpy restatement of its operation order (bit for bit) and
against a complex-step derivative (to 32 ulp); and the registration rules of the version-2 launch table."""
import ctypes as C

import numpy as np
import pytest

import user_jacobian_lib as UJ
from parallelnonlinearoptimizationlibrary_b200 import capi, problems

EPS = 2.0 ** -52


def np_lorentz_grad(a, c, w, t):
    """lorentz_term_grad in the header's order, elementwise over t[:, None] and (a, c)[None, :]"""
    with np.errstate(over="ignore", under="ignore", invalid="ignore"):
        d = t[:, None] - c[None, :]
        q = d * d
        e = w * q
        den = 1.0 + e
        u = 1.0 / den
        ja = -u
        jc = -((a[None, :] * u) * u * ((w + w) * d))
    J = np.empty((t.size, 2 * a.size))
    J[:, 0::2], J[:, 1::2] = ja, jc
    return J


def cs_jacobian(resid, x, h=1e-200):
    """complex-step derivative: J[:, j] = Im r(x + i h e_j) / h"""
    cols = []
    for j in range(x.size):
        xc = x.astype(np.complex128)
        xc[j] += 1j * h
        cols.append(np.imag(resid(xc)) / h)
    return np.stack(cols, axis=1)


def assert_within_ulps(J, Jref, ulps=32):
    scale = np.maximum(np.abs(Jref), np.max(np.abs(Jref), axis=0, keepdims=True))
    bad = np.abs(J - Jref) > ulps * EPS * scale
    assert not bad.any(), (np.argwhere(bad)[:5], J[bad][:5], Jref[bad][:5])


@pytest.fixture(scope="module")
def user():
    return UJ.build_and_load()


def test_user_jacobian_models_compile_out_of_tree_and_register(user):
    lib = capi.load_library()
    assert user.my_jacobians_registration_status() == 0
    for kind in (UJ.MYJ_F_LORENTZ, UJ.MYJ_F_GAUSS, UJ.MYJ_F_GAUSS_V1, UJ.MYJ_F_GAUSS_NOJAC):
        assert lib.pnol_functor_registered(kind) == 1


@pytest.mark.parametrize("K", [1, 2, 8, 32])
def test_lorentz_jacobian_host_is_the_header_operation_order(user, K):
    pr = problems.lorentz_problem(777, K)
    x = pr["x0"]
    for kind in (capi.F_LORENTZ_SUM, UJ.MYJ_F_LORENTZ):
        J, F = UJ.host_jacobian(kind, (pr["w"],), (pr["t"], pr["y"]), x)
        assert np.array_equal(J, np_lorentz_grad(x[0::2], x[1::2], pr["w"], pr["t"]))
    # rows far from every centre: w d^2 near the top of the range (den -> 2^1020 .. inf, u subnormal or 0) and exactly at a centre
    w = 1e300
    t = np.array([0.0, 1e2, 1e4, 1.4e4, 3e4, 1e5, -1e4, 0.5, 1e-160, 7e3])
    a, c = np.array([1.5, -2.0, 3e-3, 1e200]), np.array([0.0, 0.5, -1e-3, 2.0])
    x = np.empty(8)
    x[0::2], x[1::2] = a, c
    Jn = np_lorentz_grad(a, c, w, t)
    with np.errstate(under="ignore"):
        assert np.any((Jn != 0) & (np.abs(Jn) < np.finfo(float).tiny))       # subnormal entries are covered
    for kind in (capi.F_LORENTZ_SUM, UJ.MYJ_F_LORENTZ):
        J, _ = UJ.host_jacobian(kind, (w,), (t, np.zeros_like(t)), x)
        assert np.array_equal(J, Jn, equal_nan=True)


def test_cubic_jacobian_host_is_the_header_operation_order(user):
    rng = np.random.default_rng(3)
    xs = np.concatenate([rng.uniform(-3, 3, 500), [0.0, -0.0, 1e-170, 1e100, -7.5]])
    x3 = xs ** 3
    y = rng.normal(size=xs.size)
    J, _ = UJ.host_jacobian(capi.F_CUBIC, (), (x3, xs, y), np.array([1.0, -2.0, 0.5, 3.0]))
    want = np.stack([-x3, -(xs * xs), -xs, np.full(xs.size, -1.0)], axis=1)
    assert np.array_equal(J, want)


def _lorentz_cs(pr):
    t, y, w = pr["t"], pr["y"], pr["w"]

    def r(xc):
        a, c = xc[0::2], xc[1::2]
        return y - np.sum(a[None, :] / (1.0 + w * (t[:, None] - c[None, :]) ** 2), axis=1)
    return r


def test_every_model_matches_a_complex_step_derivative(user):
    rng = np.random.default_rng(11)
    # sum of Lorentzians, built in and the user's copy
    pr = problems.lorentz_problem(600, 16)
    Jcs = cs_jacobian(_lorentz_cs(pr), pr["x0"])
    for kind in (capi.F_LORENTZ_SUM, UJ.MYJ_F_LORENTZ):
        J, _ = UJ.host_jacobian(kind, (pr["w"],), (pr["t"], pr["y"]), pr["x0"])
        assert_within_ulps(J, Jcs)
    # exponential curve y - (x0 exp(x1 t) + x2)
    t = np.linspace(-2.0, 3.0, 400)
    y = 1.5 * np.exp(0.7 * t) + 0.2 + 0.01 * rng.normal(size=t.size)
    x = np.array([1.3, 0.65, 0.1])
    J, _ = UJ.host_jacobian(capi.F_EXPCURVE, (), (t, y), x)
    assert_within_ulps(J, cs_jacobian(lambda xc: y - (xc[0] * np.exp(xc[1] * t) + xc[2]), x))
    # cubic y - (x0 x^3 + x1 x^2 + x2 x + x3)
    xs = rng.uniform(-3, 3, 400)
    y = rng.normal(size=xs.size)
    x = np.array([0.5, -1.0, 2.0, 0.25])
    J, _ = UJ.host_jacobian(capi.F_CUBIC, (), (xs ** 3, xs, y), x)
    assert_within_ulps(J, cs_jacobian(lambda xc: y - (xc[0] * xs ** 3 + xc[1] * (xs * xs) + xc[2] * xs + xc[3]), x))
    # the user's Gaussian peak y - (A exp(-(t - mu)^2 s) + c0)
    t = np.linspace(-3.0, 5.0, 500)
    y = 2.5 * np.exp(-(t - 1.2) ** 2 * 0.8) + 0.3
    x = np.array([2.2, 1.05, 0.9])
    J, _ = UJ.host_jacobian(UJ.MYJ_F_GAUSS, (0.3,), (t, y), x)
    assert_within_ulps(J, cs_jacobian(lambda xc: y - (xc[0] * np.exp(-((t - xc[1]) ** 2) * xc[2]) + 0.3), x))


class VtableV2(C.Structure):
    """pnol_functor_vtable, ABI 2 (include/pnol_b200.h); a version-1 table is the same without the last field"""
    _fields_ = [("abi_version", C.c_int), ("n_columns", C.c_int), ("eval_batch", C.c_void_p), ("fd_points", C.c_void_p),
                ("fd_hessian", C.c_void_p), ("alpha_pool", C.c_void_p), ("residual", C.c_void_p), ("fd_jacobian", C.c_void_p),
                ("jacobian", C.c_void_p)]


def _table(abi, scalar, jacobian):
    lib = capi.load_library()
    fn = C.cast(lib.pnol_version, C.c_void_p).value        # any non-NULL code address: registration never calls a launcher
    vt = VtableV2()
    vt.abi_version, vt.n_columns = abi, 2
    if scalar:
        vt.eval_batch = vt.fd_points = vt.fd_hessian = vt.alpha_pool = fn
    else:
        vt.residual = vt.fd_jacobian = fn
    vt.jacobian = fn if jacobian else None
    return vt


def test_register_functor_version_rules():
    lib = capi.load_library()
    S, R = capi.F_USER_SCALAR_BASE + 600, capi.F_USER_RESIDUAL_BASE + 600
    # version 1: read up to fd_jacobian only. The word behind it (here non-NULL) is not the table's: a scalar kind is accepted
    # although that word, read as `jacobian`, would make it refused
    assert lib.pnol_register_functor(S, C.byref(_table(1, True, True))) == capi.PNOL_OK
    assert lib.pnol_register_functor(R, C.byref(_table(1, False, True))) == capi.PNOL_OK
    # version 2 with and without jacobian
    assert lib.pnol_register_functor(R + 1, C.byref(_table(2, False, True))) == capi.PNOL_OK
    assert lib.pnol_register_functor(R + 2, C.byref(_table(2, False, False))) == capi.PNOL_OK
    assert lib.pnol_register_functor(S + 1, C.byref(_table(2, True, False))) == capi.PNOL_OK
    # a scalar kind with an analytic Jacobian, version 0 (the 256-byte zero buffer) and unknown versions are refused
    assert lib.pnol_register_functor(S + 2, C.byref(_table(2, True, True))) == capi.ERR_INVALID
    for abi in (0, 3, -1):
        assert lib.pnol_register_functor(R + 3, C.byref(_table(abi, False, True))) == capi.ERR_INVALID
    buf = (C.c_char * 256)()
    assert lib.pnol_register_functor(R + 3, C.byref(buf)) == capi.ERR_INVALID
    for kind, want in ((S, 1), (R, 1), (R + 1, 1), (R + 2, 1), (S + 1, 1), (S + 2, 0), (R + 3, 0)):
        assert lib.pnol_functor_registered(kind) == want, kind
