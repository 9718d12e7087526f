"""GPU: every entry point that takes a functor refuses one of the other family with the status and text it has always given. A refusal
from the functor's kind says which kind, and its status depends on where the kind comes from: PNOL_ERR_NO_FUNCTOR for a built-in kind,
PNOL_ERR_INVALID for a user kind. The LM entry points that check the family by kind range themselves answer PNOL_ERR_INVALID with
their own text."""
import ctypes as C

import numpy as np
import pytest

import user_functor_lib as U
from parallelnonlinearoptimizationlibrary_b200 import capi

pytestmark = pytest.mark.gpu

N, M = 4, 64


@pytest.fixture(scope="module")
def functors(ctx):
    U.build_and_load()
    t = np.linspace(0.0, 1.0, M)
    y = np.exp(-t)
    return {
        "builtin scalar": ctx.functor(capi.F_ROSENBROCK),
        "user scalar": ctx.functor(U.MY_F_TRID, (1.0,)),
        "builtin residual": ctx.functor(capi.F_EXPCURVE, (), (), (t, y), M),
        "user residual": ctx.functor(U.MY_F_GAUSSFIT, (0.5,), (), (t, y), M),
    }


def _p(a):
    return C.c_void_p(a.ctypes.data)


def _scalar_calls(lib, h, f):
    """(entry point, status) of every scalar-objective entry point on host buffers"""
    x, dx, p = np.full(N, 0.5), np.full(N, 1e-6), np.full(N, -0.1)
    out, big = np.zeros(N), np.zeros(N * N)
    const_x, const_ind = np.zeros(N), np.zeros(N, dtype=np.uint8)
    alpha, phi, dphi = np.array([0.0, 0.5, 1.0]), np.zeros(3), np.zeros(3)
    f0, bad = C.c_double(), C.c_int()
    pts = np.full((8, N), 0.25)
    yield "eval_batch", lib.pnol_eval_batch(h, f, _p(pts), C.c_longlong(8), N, C.c_longlong(N), None, _p(out))
    yield "eval_recur", lib.pnol_eval_recur(h, f, _p(x), N, _p(const_x), _p(const_ind), N, C.byref(f0))
    yield "fd_gradient", lib.pnol_fd_gradient(h, f, _p(x), _p(dx), N, _p(out), C.byref(f0))
    yield "fd_gradient_recur", lib.pnol_fd_gradient_recur(h, f, _p(x), _p(dx), N, _p(const_x), _p(const_ind), N, _p(out), C.byref(f0))
    yield "gradient", lib.pnol_gradient(h, f, _p(x), N, _p(out), None)
    yield "gradient_recur", lib.pnol_gradient_recur(h, f, _p(x), N, _p(const_x), _p(const_ind), N, _p(out), None)
    yield "fd_hessian", lib.pnol_fd_hessian(h, f, _p(x), _p(dx), N, _p(big))
    yield "hessian", lib.pnol_hessian(h, f, _p(x), N, _p(big))
    yield "alpha_pool", lib.pnol_alpha_pool(h, f, _p(x), _p(p), N, _p(alpha), 3, C.c_double(1e-8), None, None, None, N, _p(phi), _p(dphi),
                                            C.byref(bad))
    yield "alpha_pool_analytic", lib.pnol_alpha_pool_analytic(h, f, _p(x), _p(p), N, _p(alpha), 3, None, None, None, N, _p(phi), _p(dphi),
                                                              C.byref(bad))


def _residual_calls(ctx, lib, h, f):
    """(entry point, status) of every residual-model entry point; the LM steps take device buffers"""
    x, dx = np.full(N, 0.5), np.full(N, 1e-6)
    J, F, nn, v = np.zeros(M * N), np.zeros(M), np.zeros(N * N), np.zeros(N)
    ss = C.c_double()
    for mode in (capi.JAC_AUTO, capi.JAC_BLACKBOX, capi.JAC_STRUCTURED, capi.JAC_ANALYTIC):
        yield "fd_jacobian mode %d" % mode, lib.pnol_fd_jacobian(h, f, _p(x), _p(dx), N, _p(J), _p(F), mode)
    yield "residual_eval", lib.pnol_residual_eval(h, f, _p(x), N, _p(F), C.byref(ss))
    yield "lm_normal_eq_fused", lib.pnol_lm_normal_eq_fused(h, f, _p(x), _p(dx), N, C.c_double(1e-3), _p(nn), _p(nn), _p(v), _p(F))
    dev = [ctx.malloc(8 * M * N) for _ in range(4)]
    try:
        dJ, dF, dFt, dJTJ = (C.c_void_p(d) for d in dev)
        sigma, xt, info = np.zeros(N), np.zeros(N), C.c_int()
        yield "lm_step", lib.pnol_lm_step(h, f, _p(x), _p(dx), N, dJ, dF, dFt, C.c_double(1e-3), capi.JAC_AUTO, 0, dJTJ, _p(sigma), _p(xt),
                                          C.byref(ss), C.byref(info))
        lam, chi, acc, rej, sw = C.c_double(1e-3), C.c_double(1.0), C.c_int(), C.c_int(), C.c_int()
        yield "lm_iterate", lib.pnol_lm_iterate(h, f, _p(x), _p(dx), N, dJ, dF, dFt, dJTJ, C.byref(lam), C.byref(chi), C.c_double(10.0),
                                                C.c_double(0.0), 1, capi.JAC_AUTO, C.byref(acc), C.byref(rej), C.byref(sw))
    finally:
        for d in dev:
            ctx.free(d)
    ro, X = np.array([0, M], dtype=np.int64), np.full((1, N), 0.5)
    chisq, lam_b, it, stp = np.zeros(1), np.zeros(1), np.zeros(1, dtype=np.int32), np.zeros(1, dtype=np.int32)
    yield "lm_batch", lib.pnol_lm_batch(h, f, _p(ro), C.c_longlong(1), N, _p(X), _p(dx), C.c_double(1e-3), C.c_double(10.0),
                                        C.c_double(1e-7), 10, capi.JAC_AUTO, _p(chisq), _p(lam_b), _p(it), _p(stp), None)


@pytest.mark.parametrize("origin", ["builtin", "user"])
def test_scalar_entry_points_refuse_a_residual_model(ctx, functors, origin):
    f = functors[origin + " residual"]
    want = capi.ERR_NO_FUNCTOR if origin == "builtin" else capi.ERR_INVALID
    text = "functor kind %d is not a scalar objective" % f.kind
    for name, st in _scalar_calls(ctx.lib, ctx.h, f.handle):
        assert (st, ctx.lib.pnol_last_error(ctx.h).decode()) == (want, text), name
    ga = ctx.ga_create(f, N, np.full(N, -1.0), np.full(N, 1.0), 64, 2, dict(seed=1))
    try:
        st = ctx.lib.pnol_ga_init(ga.handle, _p(np.zeros(N)), None)
        assert (st, ctx.lib.pnol_last_error(ctx.h).decode()) == (want, text), "ga_init"
    finally:
        ga.close()


@pytest.mark.parametrize("origin", ["builtin", "user"])
def test_residual_entry_points_refuse_a_scalar_objective(ctx, functors, origin):
    f = functors[origin + " scalar"]
    family = (capi.ERR_NO_FUNCTOR if origin == "builtin" else capi.ERR_INVALID, "functor kind %d is not a residual model" % f.kind)
    want = {
        "fd_jacobian mode %d" % capi.JAC_AUTO: family,
        "fd_jacobian mode %d" % capi.JAC_BLACKBOX: family,
        "fd_jacobian mode %d" % capi.JAC_STRUCTURED: (capi.ERR_NO_FUNCTOR, "functor kind %d has no structured Jacobian for n = %d" % (f.kind, N)),
        "fd_jacobian mode %d" % capi.JAC_ANALYTIC: family,
        "residual_eval": family,
        "lm_normal_eq_fused": (capi.ERR_INVALID, "lm_normal_eq_fused: the functor is not a residual model"),
        "lm_step": (capi.ERR_INVALID, "lm_step: the functor is not a residual model"),
        "lm_iterate": (capi.ERR_INVALID, "lm_iterate: the functor is not a residual model"),
        "lm_batch": (capi.ERR_INVALID, "lm_batch: functor kind %d is not a residual model" % f.kind),
    }
    got = {}
    for name, st in _residual_calls(ctx, ctx.lib, ctx.h, f.handle):
        got[name] = (st, ctx.lib.pnol_last_error(ctx.h).decode())
    assert got == want
