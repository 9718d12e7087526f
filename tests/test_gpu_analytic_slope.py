"""GPU: analytic line-search slopes (pnol_alpha_pool_analytic) against the host restatement bit for bit -- phi from the CPU stand-in
(tests/host_logic_standin.cpp) and from pnol_alpha_pool, the slope from the functor's host partial() summed as dotProd sums
(tests/test_user_slope_cpu.py) -- for every built-in and both user kinds of tests/user_functor/my_gradients.hpp, up to the largest n
pnol_alpha_pool accepts; the slope at alpha = 0 against dotProd(pnol_gradient[_recur], p); the sentinel; the refusals; and BFGS, BFGS_Bnd
and BFGS_Bnd_MPI_SW with Runtime::setAnalyticSlope(true) against the same controllers on the stand-in."""
import ctypes as C

import numpy as np
import pytest

import host_standin
import test_user_slope_cpu as SC
import user_functor_lib as UF
import user_gradient_lib as UG
from parallelnonlinearoptimizationlibrary_b200 import capi

pytestmark = pytest.mark.gpu
CASES = SC.CASES


def _nmax():
    """the largest n pnol_alpha_pool accepts: n * 17 + 16 bytes of opt-in shared memory (13672 on a B200)"""
    import torch
    return (int(torch.cuda.get_device_properties(0).shared_memory_per_block_optin) - 16) // 17


@pytest.fixture(scope="module")
def user():
    return UG.build_and_load()


@pytest.fixture(scope="module")
def standin():
    hl = host_standin.load()
    if hl is None:
        pytest.skip("no g++ on this box")
    return SC.Standin(hl)


def _functor(ctx, name):
    kind, sc, ints, cols, _, _ = CASES[name]
    return ctx.functor(kind, sc, ints, cols, cols[0].size if cols else 0)


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def _same(a, b):
    return np.array_equal(_bits(a), _bits(b))


def _sizes(name):
    fixed = CASES[name][4]
    return [fixed] if fixed else [1, 2, 3, 31, 32, 33, 127, 128, 129, 1000, 4096, _nmax()]


def _check(ctx, standin, f, sf, name, x, p, alpha, cx=None, ci=None):
    """device vs host: phi (stand-in for built-ins, pnol_alpha_pool always) and the slope (numpy over the host partial())"""
    phi, dphi, bad = ctx.alpha_pool_analytic(f, x, p, alpha, const_x=cx, const_ind=ci)
    assert bad == 0
    assert _same(dphi, SC.py_slopes(name, x, p, alpha, cx, ci)), name
    assert _same(phi, ctx.alpha_pool(f, x, p, alpha, 1e-6, const_x=cx, const_ind=ci)[0]), name
    if sf is not None:
        want = standin.pool(sf, x, p, alpha, const_x=cx, const_ind=ci)
        assert _same(phi, want[0]) and _same(dphi, want[1]), name
    return phi, dphi


@pytest.mark.parametrize("name", sorted(CASES))
def test_slopes_are_the_host_restatement_bit_for_bit(ctx, user, standin, name):
    import torch
    rng = np.random.default_rng(len(name))
    f = _functor(ctx, name)
    sf = standin.functor(name) if name in SC.BUILTIN_CASES else None
    for n in _sizes(name):
        x, p = SC._x(name, n, rng), rng.normal(size=n)
        alpha = SC.ALPHAS if n <= 4096 else SC.ALPHAS[:3]
        phi, dphi = _check(ctx, standin, f, sf, name, x, p, alpha)
        if n >= 3:
            # an active set, with as many reduced entries as free variables and with more (those give 0 * p_r)
            nfull = n + 2 if n + 2 <= _nmax() else n
            ci = np.zeros(nfull, np.uint8)
            ci[1::3] = 1
            cx = rng.uniform(-1, 1, nfull)
            free = int((ci == 0).sum())
            for nr in (free, min(free + 2, nfull)):
                _check(ctx, standin, f, sf, name, SC._x(name, nr, rng), rng.normal(size=nr), alpha[:4], cx, ci)
        if n in (33, 4096):
            # an eval_ind mask (masked entries keep the caller's values), device pointers, x misaligned by one double
            ei = (np.arange(alpha.size) % 3 != 1).astype(np.uint8)
            xb = torch.empty(n + 1, dtype=torch.float64, device="cuda")
            xb[1:] = torch.from_numpy(x).cuda()
            pd, ad = torch.from_numpy(p).cuda(), torch.from_numpy(alpha).cuda()
            phd = torch.full((alpha.size,), -7.0, dtype=torch.float64, device="cuda")
            dpd = torch.full((alpha.size,), -7.0, dtype=torch.float64, device="cuda")
            torch.cuda.synchronize()
            ctx.alpha_pool_analytic(f, xb.data_ptr() + 8, pd, ad, eval_ind=ei, phi=phd, dphi=dpd, n=n, npool=alpha.size)
            ph, dp = phd.cpu().numpy(), dpd.cpu().numpy()
            assert _same(ph[ei == 1], phi[ei == 1]) and _same(dp[ei == 1], dphi[ei == 1]), (name, n)
            assert np.all(ph[ei == 0] == -7.0) and np.all(dp[ei == 0] == -7.0), (name, n)
    f.close()


@pytest.mark.parametrize("name", sorted(CASES))
def test_slope_at_zero_is_dotprod_of_the_analytic_gradient(ctx, user, name):
    """alpha = 0, finite p, no -0 in x: the slope is dotProd(pnol_gradient(x), p), and with an active set
    dotProd(pnol_gradient_recur(...), p), bit for bit -- the host's dphi0dalpha"""
    rng = np.random.default_rng(3 + len(name))
    f = _functor(ctx, name)
    for n in _sizes(name):
        x, p = SC._x(name, n, rng), rng.normal(size=n)
        _, dphi, _ = ctx.alpha_pool_analytic(f, x, p, [0.0])
        assert _same(dphi[0], SC.seq_dot(ctx.gradient(f, x)[0], p)), (name, n)
        if n >= 3 and n < _nmax():
            ci = np.zeros(n + 1, np.uint8)
            ci[::4] = 1
            cx = rng.uniform(-1, 1, n + 1)
            for nr in (int((ci == 0).sum()), int((ci == 0).sum()) + 1):
                xr, pr = SC._x(name, nr, rng), rng.normal(size=nr)
                _, dphi, _ = ctx.alpha_pool_analytic(f, xr, pr, [0.0], const_x=cx, const_ind=ci)
                assert _same(dphi[0], SC.seq_dot(ctx.gradient_recur(f, xr, cx, ci)[0], pr)), (name, n, nr)
    f.close()


def test_nan_and_inf_phi_become_the_sentinel_and_the_slope_stays_raw(ctx):
    f = ctx.functor(capi.F_ROSENBROCK)
    x, p = np.array([0.5, 1e200, 0.3, -0.2]), np.array([1.0, 1.0, -1.0, 0.5])
    alpha = np.array([0.0, 1.0, np.nan])
    phi, dphi, bad = ctx.alpha_pool_analytic(f, x, p, alpha)
    phi_fd, _, bad_fd = ctx.alpha_pool(f, x, p, alpha, 1e-6)
    assert bad == bad_fd == 3 and np.all(phi == 1e10) and _same(phi, phi_fd)
    # raw slopes: the host's values, a NaN wherever the host has one (NaN payloads may differ between host and device)
    want = SC.py_slopes("rosenbrock", x, p, alpha)
    assert np.isnan(dphi[2]) and np.array_equal(np.isnan(dphi), np.isnan(want))
    assert _same(dphi[~np.isnan(want)], want[~np.isnan(want)])
    f.close()


def test_refusals(ctx, user):
    import torch
    lib = ctx.lib
    UF.build_and_load()
    x, p, a, ph, dp = np.full(4, 0.5), np.ones(4), np.array([0.0, 1.0]), np.empty(2), np.empty(2)

    def call(fh, n=4, xx=x, dphi=dp):
        return lib.pnol_alpha_pool_analytic(ctx.h, fh, capi._ptr(xx), capi._ptr(p), n, capi._ptr(a), 2, None, None, None, n,
                                            capi._ptr(ph), capi._ptr(dphi), None)
    # a user scalar objective without partial(): refused, never a forward difference; the error names the kind
    ft = ctx.functor(UF.MY_F_TRID)
    assert call(ft.handle) == capi.ERR_NO_FUNCTOR
    assert str(UF.MY_F_TRID).encode() in lib.pnol_last_error(ctx.h) and b"partial" in lib.pnol_last_error(ctx.h)
    ft.close()
    # residual models: refused as pnol_alpha_pool refuses them
    t, y = SC._t_y()
    for fr in (ctx.functor(capi.F_EXPCURVE, (), (), (t, y), t.size), ctx.functor(UF.MY_F_GAUSSFIT, (0.3,), (), (t, y), t.size)):
        st = call(fr.handle, 3)
        st_fd = lib.pnol_alpha_pool(ctx.h, fr.handle, capi._ptr(x), capi._ptr(p), 3, capi._ptr(a), 2, C.c_double(1e-6), None, None, None, 3,
                                    capi._ptr(ph), capi._ptr(dp), None)
        assert st == st_fd != capi.PNOL_OK
        fr.close()
    fr = ctx.functor(capi.F_ROSENBROCK)
    assert call(fr.handle, dphi=None) == capi.ERR_INVALID                              # dphi is required
    # n beyond the range: the point and the products do not fit in shared memory (device buffers: nothing is staged)
    optin = int(torch.cuda.get_device_properties(0).shared_memory_per_block_optin)
    n = optin // 16 + 1
    xd = torch.full((n,), 0.5, dtype=torch.float64, device="cuda")
    pd = torch.ones(n, dtype=torch.float64, device="cuda")
    st = lib.pnol_alpha_pool_analytic(ctx.h, fr.handle, capi._ptr(xd), capi._ptr(pd), n, capi._ptr(a), 2, None, None, None, n,
                                      capi._ptr(ph), capi._ptr(dp), None)
    assert st == capi.ERR_INVALID and b"shared memory" in lib.pnol_last_error(ctx.h)
    fr.close()


# ---- the plugin classes ----
@pytest.fixture
def host(ctx):
    from parallelnonlinearoptimizationlibrary_b200 import hostapi
    hostapi.attach(ctx)
    yield hostapi
    hostapi.set_analytic_gradient(False)
    hostapi.set_analytic_slope(False)
    hostapi.set_hinv_mode(capi.HINV_RANK2)
    hostapi.detach()


def _run(host, variant, obj, x0, iters, dalpha=1e-6):
    bounded = variant in ("bfgs_bnd", "bfgs_bnd_sw")
    lb, ub = (np.full(x0.size, -5.0), np.full(x0.size, 5.0)) if bounded else (None, None)
    return host.bfgs(variant, obj, x0, SC.bfgs_params(variant, iters, dalpha), lb, ub, pool_width=SC.VARIANTS[variant])


@pytest.mark.parametrize("variant", SC.SLOPED)
def test_bfgs_with_analytic_slopes_reaches_the_optimum(host, variant):
    host.set_analytic_gradient(True)
    host.set_analytic_slope(True)
    for obj, x0, xopt, fopt in SC.PROBLEMS:
        r = _run(host, variant, obj, x0, 1000, dalpha=np.nan)          # dalpha = NaN: no forward difference is taken
        assert np.linalg.norm(r["X"] - xopt) <= 1e-4 * max(np.linalg.norm(xopt), 1.0), (obj, r)
        assert abs(r["fOpt"] - fopt) < 1e-8, (obj, r)


@pytest.mark.parametrize("variant", SC.SLOPED)
@pytest.mark.parametrize("obj", ["rosenbrock", "booth", "goldstein"])
def test_bfgs_iterates_match_the_host_logic_stand_in(host, standin, variant, obj):
    """Analytic gradient and slopes. The stand-in runs the same host controllers with the host partials and the dense algebra on the
    CPU, in the literal two-product updateHessianInv; the GPU is set to the same form. What remains is the summation order of the
    device's dense algebra (DESIGN 2)."""
    import test_host_logic_cpu as TH
    hl = standin.lib
    x0 = {p[0]: p[1] for p in SC.PROBLEMS}[obj]
    iters = 1 if obj == "booth" else 5        # Booth: a quadratic, the first step lands on the optimum up to rounding
    host.set_hinv_mode(capi.HINV_LITERAL)
    host.set_analytic_gradient(True)
    host.set_analytic_slope(True)
    with SC.modes(hl):
        b = SC.run_bfgs(hl, variant, obj, x0, iters)
    a = _run(host, variant, obj, x0, iters)
    assert a["iterations"] == b["iterations"]
    assert np.linalg.norm(a["X"] - b["X"]) <= 1e-9 * np.linalg.norm(b["X"]), (a["X"], b["X"])
    assert abs(a["fOpt"] - b["fOpt"]) <= 1e-9 * max(abs(b["fOpt"]), 1e-300) or a["fOpt"] == b["fOpt"]


def test_pool_member_counts_one_evaluation_per_entry(host, standin):
    rng = np.random.default_rng(5)
    x, p = rng.uniform(-2, 2, 10), rng.normal(size=10)
    ci = np.zeros(12, np.uint8)
    ci[[3, 7]] = 1
    cx = rng.uniform(-1, 1, 12)
    sf = standin.functor("rosenbrock")
    phi, dphi, ev = SC.pool_member(host.lib(), "rosenbrock", x, p, SC.ALPHAS, cx, ci)
    assert ev == 2 * SC.ALPHAS.size
    host.set_analytic_slope(True)
    phi_a, dphi_a, ev_a = SC.pool_member(host.lib(), "rosenbrock", x, p, SC.ALPHAS, cx, ci)
    assert ev_a == SC.ALPHAS.size
    want = standin.pool(sf, x, p, SC.ALPHAS, const_x=cx, const_ind=ci)
    assert _same(phi_a, want[0]) and _same(dphi_a, want[1]) and _same(phi_a, phi)
