"""Analytic line-search slopes (pnol_alpha_pool_analytic) without a GPU: the CPU stand-in extended by the slope
(tests/host_logic_slope.cpp: the host eval() and partial() of include/pnol/functors.hpp with the kernel's point assembly, sequential sum
and sentinel) against dotProd of its own pnol_gradient_recur at alpha = 0 (bit for bit), against a numpy restatement over the host
partial() of every built-in and of the user's tests/user_functor/my_gradients.hpp (bit for bit), and against a complex-step or mpmath
directional derivative; the registration rules of pnol_register_functor_slope; and the BFGS controllers with
Runtime::setAnalyticSlope(true) on the CPU."""
import ctypes as C

import mpmath
import numpy as np
import pytest

import host_logic_slope_lib as HLS
import user_gradient_lib as UG
import user_hessian_lib as UH
from parallelnonlinearoptimizationlibrary_b200 import capi

EPS = 2.0 ** -52
SCALAR_BUILTINS = (capi.F_ROSENBROCK, capi.F_POWER, capi.F_BOOTH, capi.F_GOLDSTEIN, capi.F_RASTRIGIN, capi.F_EXPCURVE_SINGLE)
ULPS = 64          # accuracy bound of a slope, in units of EPS * sum_r |p_r g_r| (n = 40 terms summed sequentially)


def _t_y():
    t = np.linspace(-2.0, 3.0, 257)
    return t, 1.5 * np.exp(0.7 * t) + 0.2 + 0.01 * np.sin(7 * t)


# name: kind, scalars, ints, columns, n of the tests (0: any), start-point scale
CASES = {
    "rosenbrock": (capi.F_ROSENBROCK, (), (), (), 0, 2.0),
    "power3": (capi.F_POWER, (), (3,), (), 0, 2.0),
    "booth": (capi.F_BOOTH, (), (), (), 2, 3.0),
    "goldstein": (capi.F_GOLDSTEIN, (), (), (), 2, 2.0),
    "rastrigin": (capi.F_RASTRIGIN, (), (), (), 0, 5.12),
    "expsingle": (capi.F_EXPCURVE_SINGLE, (), (), _t_y(), 3, 1.0),
    "user_trid": (UG.MYG_F_TRID, (), (), (), 0, 2.0),
    "user_styblinski": (UG.MYG_F_STYBLINSKI, (0.5,), (), (), 0, 4.0),
}
BUILTIN_CASES = [k for k, v in CASES.items() if v[0] < capi.F_USER_SCALAR_BASE]


@pytest.fixture(scope="module")
def user():
    return UG.build_and_load()


@pytest.fixture(scope="module")
def standin():
    hl = HLS.build_and_load()
    if hl is None:
        pytest.skip("no g++ on this box")
    return Standin(hl)


def _p(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


class Standin:
    """the C-ABI entry points of the extended stand-in, called directly"""

    def __init__(self, lib):
        self.lib = lib
        c = C.c_void_p()
        assert lib.pnol_ctx_create(C.byref(c), 0) == 0
        self.ctx = c
        self._keep = []

    def functor(self, name):
        kind, sc, ints, cols, _, _ = CASES[name]
        d = capi.FunctorDesc()
        d.kind = kind
        for i, v in enumerate(sc):
            d.scalars[i] = float(v)
        for i, v in enumerate(ints):
            d.ints[i] = int(v)
        d.n_columns = len(cols)
        for i, c in enumerate(cols):
            c = np.ascontiguousarray(c, dtype=np.float64)
            self._keep.append(c)
            d.columns[i] = c.ctypes.data
        d.m = cols[0].size if cols else 0
        f = C.c_void_p()
        assert self.lib.pnol_functor_create(self.ctx, C.byref(d), C.byref(f)) == 0
        return f

    def pool(self, f, x, p, alpha, eval_ind=None, const_x=None, const_ind=None, phi=None, dphi=None):
        x, p, alpha = (np.ascontiguousarray(a, dtype=np.float64) for a in (x, p, alpha))
        phi = np.zeros(alpha.size) if phi is None else phi.copy()
        dphi = np.zeros(alpha.size) if dphi is None else dphi.copy()
        ei = None if eval_ind is None else np.ascontiguousarray(eval_ind, dtype=np.uint8)
        cx = None if const_x is None else np.ascontiguousarray(const_x, dtype=np.float64)
        ci = None if const_ind is None else np.ascontiguousarray(const_ind, dtype=np.uint8)
        bad = C.c_int()
        st = self.lib.pnol_alpha_pool_analytic(self.ctx, f, _p(x), _p(p), x.size, _p(alpha), alpha.size, _p(ei), _p(cx), _p(ci),
                                               x.size if cx is None else cx.size, _p(phi), _p(dphi), C.byref(bad))
        assert st == 0
        return phi, dphi, bad.value

    def gradient_recur(self, f, xr, const_x, const_ind):
        xr = np.ascontiguousarray(xr, dtype=np.float64)
        g = np.empty(xr.size)
        ci = np.ascontiguousarray(const_ind, dtype=np.uint8)
        assert self.lib.pnol_gradient_recur(self.ctx, f, _p(xr), xr.size, _p(np.ascontiguousarray(const_x, dtype=np.float64)), _p(ci), ci.size,
                                            _p(g), None) == 0
        return g


def seq_dot(g, p):
    """dotProd (include/pnol/UtilityFunctions.hpp): s = 0; s = s + g[r] * p[r] in r order"""
    s = 0.0
    for a, b in zip(g.tolist(), p.tolist()):
        s = s + a * b
    return s


def assemble(x, p, const_x, const_ind):
    """the full point, the full direction and the slot of every reduced entry, as the library assembles them"""
    if const_ind is None:
        return x.copy(), p.copy(), np.arange(x.size, dtype=np.int32)
    nfull = const_ind.size
    xf, pf, pos = np.zeros(nfull), np.zeros(nfull), np.full(x.size, -1, dtype=np.int32)
    k = 0
    for j in range(nfull):
        if const_ind[j]:
            xf[j] = const_x[j]
            continue
        if k < x.size:
            xf[j], pf[j], pos[k] = x[k], p[k], j
        k += 1
    return xf, pf, pos


def py_slopes(name, x, p, alpha, const_x=None, const_ind=None):
    """the slope of every pool entry restated in numpy over the functor's host partial() (tests/user_gradient_lib.py)"""
    kind, sc, ints, cols, _, _ = CASES[name]
    xf, pf, pos = assemble(x, p, const_x, const_ind)
    isc = np.zeros(xf.size, bool) if const_ind is None else const_ind.astype(bool)
    out = []
    for a in np.asarray(alpha, dtype=np.float64):
        xa = np.where(isc, xf, xf + a * pf)
        g = np.zeros(x.size)
        live = pos >= 0
        if live.any():
            g[live] = UG.host_partials(kind, xa, sc, ints, cols, idx=pos[live])
        out.append(seq_dot(g, p))
    return np.array(out)


def _same(a, b):
    """bit for bit, +0 and -0 told apart"""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return a.shape == b.shape and np.array_equal(a.view(np.int64), b.view(np.int64))


def _n(name, n):
    return CASES[name][4] or n


def _x(name, n, rng):
    x = rng.uniform(-CASES[name][5], CASES[name][5], n)
    x[x == 0] = 0.5
    return x


ALPHAS = np.array([0.0, 1e-8, 1e-3, 0.1, 0.5, 1.0, 2.0, -0.25, 3.0])


def test_user_slope_launchers_attach_exactly_with_partial(user):
    lib = capi.load_library()
    assert user.my_gradients_registration_status() == 0
    for kind in (UG.MYG_F_TRID, UG.MYG_F_STYBLINSKI):                      # partial(): gradient and slope attached
        assert lib.pnol_functor_has_gradient(kind) == 1 and lib.pnol_functor_has_slope(kind) == 1
    for kind in SCALAR_BUILTINS:
        assert lib.pnol_functor_has_slope(kind) == 1
    UH.build_and_load()
    for kind in (UH.MYH_F_QUADFORM, UH.MYH_F_STYBLINSKI):                  # partial2() only: no slope
        assert lib.pnol_functor_registered(kind) == 1 and lib.pnol_functor_has_slope(kind) == 0
    for kind in (capi.F_EXPCURVE, capi.F_CUBIC, capi.F_LORENTZ_SUM, 0, 7, capi.F_USER_SCALAR_BASE + 999):
        assert lib.pnol_functor_has_slope(kind) == 0


@pytest.mark.parametrize("name", BUILTIN_CASES)
def test_slope_at_zero_is_dotprod_of_the_gradient_recur(user, standin, name):
    """alpha = 0: the slope is dotProd(pnol_gradient_recur(x), p) bit for bit, with and without an active set and with more reduced
    entries than free variables"""
    rng = np.random.default_rng(len(name))
    for n in (1, 2, 3, 17, 40):
        n = _n(name, n)
        f = standin.functor(name)
        x, p = _x(name, n, rng), rng.normal(size=n)
        ind = np.zeros(n, np.uint8)
        phi, dphi, bad = standin.pool(f, x, p, [0.0])
        assert bad == 0 and _same(dphi[0], seq_dot(standin.gradient_recur(f, x, x, ind), p)), (name, n)
        if n >= 3:
            ind[::3] = 1
            cx = rng.uniform(-1, 1, n)
            for nr in (int((ind == 0).sum()), int((ind == 0).sum()) + 1):
                xr, pr = _x(name, nr, rng), rng.normal(size=nr)
                phi, dphi, bad = standin.pool(f, xr, pr, [0.0], const_x=cx, const_ind=ind)
                assert _same(dphi[0], seq_dot(standin.gradient_recur(f, xr, cx, ind), pr)), (name, n, nr)


@pytest.mark.parametrize("name", BUILTIN_CASES)
def test_standin_slopes_are_the_numpy_restatement(user, standin, name):
    """every pool entry, the eval_ind mask (masked entries keep the caller's values), active sets, the sentinel on phi only"""
    rng = np.random.default_rng(7 + len(name))
    n = _n(name, 12)
    f = standin.functor(name)
    x, p = _x(name, n, rng), rng.normal(size=n)
    phi, dphi, bad = standin.pool(f, x, p, ALPHAS)
    assert bad == 0 and _same(dphi, py_slopes(name, x, p, ALPHAS))
    ei = (np.arange(ALPHAS.size) % 2).astype(np.uint8)
    keep = np.full(ALPHAS.size, -7.0)
    phi2, dphi2, _ = standin.pool(f, x, p, ALPHAS, eval_ind=ei, phi=keep, dphi=keep)
    assert _same(phi2[ei == 1], phi[ei == 1]) and _same(dphi2[ei == 1], dphi[ei == 1]) and np.all(phi2[ei == 0] == -7.0) and np.all(dphi2[ei == 0] == -7.0)
    if n >= 3:
        ind = np.zeros(n, np.uint8)
        ind[1::4] = 1
        cx = rng.uniform(-1, 1, n)
        for nr in (int((ind == 0).sum()), int((ind == 0).sum()) + 2):
            xr, pr = _x(name, nr, rng), rng.normal(size=nr)
            _, dphi3, _ = standin.pool(f, xr, pr, ALPHAS, const_x=cx, const_ind=ind)
            assert _same(dphi3, py_slopes(name, xr, pr, ALPHAS, cx, ind)), (name, nr)
    # NaN / inf phi -> 1e10 and counted; the slope stays raw
    xb = x.copy()
    xb[0] = np.nan
    phi4, dphi4, bad4 = standin.pool(f, xb, p, [0.0, 1.0])
    assert bad4 == 2 and np.all(phi4 == 1e10) and np.all(np.isnan(dphi4)), (phi4, dphi4)


# ---- every slope against an independent directional derivative ----
def f_complex(name, z):
    kind, sc, ints, cols, _, _ = CASES[name]
    if name == "rosenbrock":
        return np.sum(100 * (z[1:] - z[:-1] ** 2) ** 2 + (1 - z[:-1]) ** 2)
    if name == "power3":
        return np.sum(z ** 3)
    if name == "booth":
        return (z[0] + 2 * z[1] - 7) ** 2 + (2 * z[0] + z[1] - 5) ** 2
    if name == "goldstein":
        X, Y = z[0], z[1]
        return ((1 + (X + Y + 1) ** 2 * (19 - 14 * X + 3 * X * X - 14 * Y + 6 * X * Y + 3 * Y * Y))
                * (30 + (2 * X - 3 * Y) ** 2 * (18 - 32 * X + 12 * X * X + 48 * Y - 36 * X * Y + 27 * Y * Y)))
    if name == "expsingle":
        t, y = cols
        return np.sum((y - (z[0] * np.exp(z[1] * t) + z[2])) ** 2)
    if name == "user_trid":
        return np.sum((z - 1) ** 2) - np.sum(z[1:] * z[:-1])
    if name == "user_styblinski":
        return sc[0] * np.sum(z ** 4 - 16 * z ** 2 + 5 * z)
    raise KeyError(name)


def reference_slope(name, x, p, a):
    """d/dalpha f(x + alpha p): complex step, h = 1e-200; Rastrigin (x^2 - 10 cos(2 pi x) per term): mpmath at 160 bits"""
    if name == "rastrigin":
        mpmath.mp.prec = 160
        xa = x + a * p
        return float(mpmath.fsum(mpmath.mpf(float(pr)) * (2 * mpmath.mpf(float(v)) + 20 * mpmath.pi * mpmath.sin(2 * mpmath.pi * mpmath.mpf(float(v))))
                                 for v, pr in zip(xa, p)))
    h = 1e-200
    return float(np.imag(f_complex(name, (x + a * p).astype(np.complex128) + 1j * h * p)) / h)


@pytest.mark.parametrize("name", sorted(CASES))
def test_every_slope_matches_a_complex_step_or_mpmath_derivative(user, standin, name):
    """|slope - reference| <= ULPS * EPS * sum_r |p_r g_r|"""
    kind, sc, ints, cols, _, _ = CASES[name]
    rng = np.random.default_rng(11 + len(name))
    n = _n(name, 40)
    x, p = _x(name, n, rng), rng.normal(size=n)
    alphas = np.array([0.0, 1e-3, 0.1, 0.5])
    got = py_slopes(name, x, p, alphas)
    if kind < capi.F_USER_SCALAR_BASE:
        assert _same(standin.pool(standin.functor(name), x, p, alphas)[1], got)
    for a, s in zip(alphas, got):
        g = UG.host_partials(kind, x + a * p, sc, ints, cols)
        scale = np.sum(np.abs(p * g))
        want = reference_slope(name, x, p, a)
        assert abs(s - want) <= ULPS * EPS * scale, (name, a, s, want, abs(s - want) / (EPS * scale))


# ---- registration rules (pnol_register_functor_slope) ----
def test_register_functor_slope_rules():
    from test_user_gradient_cpu import _table
    lib = capi.load_library()
    fn = C.c_void_p(C.cast(lib.pnol_version, C.c_void_p).value)      # any non-NULL code address: registration never calls a launcher
    S, R = capi.F_USER_SCALAR_BASE + 720, capi.F_USER_RESIDUAL_BASE + 720
    keep = [_table(1, True), _table(2, True), _table(2, False), _table(2, True)]
    assert lib.pnol_register_functor(S, C.byref(keep[0])) == capi.PNOL_OK          # ABI 1
    assert lib.pnol_register_functor(S + 1, C.byref(keep[1])) == capi.PNOL_OK      # ABI 2
    assert lib.pnol_register_functor(R, C.byref(keep[2])) == capi.PNOL_OK
    for kind in (S, S + 1):
        assert lib.pnol_functor_has_slope(kind) == 0
        assert lib.pnol_register_functor_slope(kind, fn) == capi.PNOL_OK
        assert lib.pnol_functor_has_slope(kind) == 1
        assert lib.pnol_functor_has_gradient(kind) == 0                            # attached separately
    assert lib.pnol_register_functor_gradient(S, fn) == capi.PNOL_OK
    assert lib.pnol_register_functor_hessian(S, fn) == capi.PNOL_OK
    # a residual kind, a kind without a table, a built-in kind, a kind outside every range and NULL are refused
    assert lib.pnol_register_functor_slope(R, fn) == capi.ERR_INVALID
    assert lib.pnol_register_functor_slope(S + 2, fn) == capi.ERR_INVALID
    assert lib.pnol_register_functor_slope(capi.F_ROSENBROCK, fn) == capi.ERR_INVALID
    assert lib.pnol_register_functor_slope(5000, fn) == capi.ERR_INVALID
    assert lib.pnol_register_functor_slope(S, None) == capi.ERR_INVALID
    assert lib.pnol_functor_has_slope(R) == 0 and lib.pnol_functor_has_slope(S + 2) == 0
    assert lib.pnol_functor_has_slope(S) == 1                                       # the refused NULL left the launcher in place
    # replacing the table drops the slope together with the gradient and the Hessian attached to the old one
    assert lib.pnol_register_functor(S, C.byref(keep[3])) == capi.PNOL_OK
    assert lib.pnol_functor_has_slope(S) == 0 and lib.pnol_functor_has_gradient(S) == 0 and lib.pnol_functor_has_hessian(S) == 0
    assert lib.pnol_functor_registered(S) == 1 and lib.pnol_functor_has_slope(S + 1) == 1


# ---- the host controllers in the analytic mode, without a GPU ----
def bfgs_params(variant, iters, dalpha=1e-6):
    """setParams of the five BFGS classes (host_capi.cpp: pnolhost_bfgs), the examples' settings; dalpha where the class has one"""
    if variant == "bfgs":
        return [1e-4, 0.9, dalpha, 1.0, 1000, 1e-7, 1e-3, iters, 1e-5, 1e-5, 0]
    if variant == "bfgs_mpi":
        return [1e-4, 0.9, 4.0, 1.0, 50, 1e-7, 1e-3, iters, 1e-5, 1e-5, 0]
    if variant == "bfgsbnd_mpi":
        return [1e-4, 0.1, 1e-16, 4.0, 1.0, 1000, 1e-7, 1e-3, iters, 1e-5, 1e-5, 1e-5, 0]
    return [1e-4, 0.8, dalpha, 1.0, 1e-10, 2.0, 50, 1e-5, 1e-6, 1e-3, iters, 1e-5, 1e-5, 0]      # bfgs_bnd, bfgs_bnd_sw


VARIANTS = {"bfgs": 0, "bfgs_mpi": 4, "bfgs_bnd": 0, "bfgs_bnd_sw": 8, "bfgsbnd_mpi": 4}        # variant: pool width
SLOPED = ("bfgs", "bfgs_bnd", "bfgs_bnd_sw")                                                    # the classes whose line searches take slopes
PROBLEMS = [("rosenbrock", np.full(10, 3.0), np.ones(10), 0.0), ("booth", np.array([3.0, -2.0]), np.array([1.0, 3.0]), 0.0),
            ("goldstein", np.array([0.1, -0.9]), np.array([0.0, -1.0]), 3.0)]


def run_bfgs(lib, variant, obj, x0, iters, dalpha=1e-6):
    import test_host_logic_cpu as TH
    bounded = variant in ("bfgs_bnd", "bfgs_bnd_sw", "bfgsbnd_mpi")
    lb, ub = (np.full(x0.size, -5.0), np.full(x0.size, 5.0)) if bounded else (None, None)
    return TH.bfgs(lib, variant, obj, x0, bfgs_params(variant, iters, dalpha), lb, ub, VARIANTS[variant])


class modes:
    """analytic gradient and, optionally, analytic slopes on a host library for the duration of a block"""

    def __init__(self, lib, slope=True):
        self.lib, self.slope = lib, slope

    def __enter__(self):
        self.lib.pnolhost_set_analytic_gradient(1)
        self.lib.pnolhost_set_analytic_slope(int(self.slope))

    def __exit__(self, *exc):
        self.lib.pnolhost_set_analytic_gradient(0)
        self.lib.pnolhost_set_analytic_slope(0)


@pytest.mark.parametrize("variant", sorted(VARIANTS))
def test_bfgs_controllers_with_analytic_slopes(standin, variant):
    """BFGS, BFGS_Bnd and BFGS_Bnd_MPI_SW reach the known optima with dalpha = NaN (no forward difference is taken); BFGS_MPI and
    BFGSBnd_MPI use values only and run as without the switch, bit for bit."""
    hl = standin.lib
    for obj, x0, xopt, fopt in PROBLEMS:
        if variant in SLOPED:
            with modes(hl):
                r = run_bfgs(hl, variant, obj, x0, 1000, dalpha=np.nan)
            assert np.linalg.norm(r["X"] - xopt) <= 1e-4 * max(np.linalg.norm(xopt), 1.0), (obj, r)
            assert abs(r["fOpt"] - fopt) < 1e-8, (obj, r)
        else:
            with modes(hl):
                r = run_bfgs(hl, variant, obj, x0, 30)
            with modes(hl, slope=False):
                r0 = run_bfgs(hl, variant, obj, x0, 30)
            assert np.array_equal(r["X"], r0["X"]) and r["fOpt"] == r0["fOpt"] and r["iterations"] == r0["iterations"], (obj, r, r0)


def pool_member(lib, obj, x, p, alpha, const_x=None, const_ind=None):
    """BFGS_Bnd_MPI_SW::evaluateAlphaPoolAndDerivatives through pnolhost_alpha_pool_sw: (phi, dphi, objective evaluations)"""
    x, p, alpha = (np.ascontiguousarray(a, dtype=np.float64) for a in (x, p, alpha))
    cx = None if const_x is None else np.ascontiguousarray(const_x, dtype=np.float64)
    ci = None if const_ind is None else np.ascontiguousarray(const_ind, dtype=np.uint8)
    phi, dphi, ev = np.empty(alpha.size), np.empty(alpha.size), C.c_longlong()
    st = lib.pnolhost_alpha_pool_sw(obj.encode(), _p(x), _p(p), x.size, _p(alpha), alpha.size, _p(cx), _p(ci), x.size if ci is None else ci.size,
                                    _p(phi), _p(dphi), C.byref(ev))
    assert st == 0, lib.pnolhost_last_error()
    return phi, dphi, ev.value


def test_pool_member_counts_one_evaluation_per_entry(standin):
    hl = standin.lib
    rng = np.random.default_rng(5)
    x, p = rng.uniform(-2, 2, 10), rng.normal(size=10)
    ind = np.zeros(12, np.uint8)
    ind[[3, 7]] = 1
    cx = rng.uniform(-1, 1, 12)
    f = standin.functor("rosenbrock")
    for c_x, c_i in ((x, np.zeros(10, np.uint8)), (cx, ind)):
        phi, dphi, ev = pool_member(hl, "rosenbrock", x, p, ALPHAS, c_x, c_i)
        assert ev == 2 * ALPHAS.size                                               # the forward difference: two per entry
        with modes(hl):
            phi_a, dphi_a, ev_a = pool_member(hl, "rosenbrock", x, p, ALPHAS, c_x, c_i)
        assert ev_a == ALPHAS.size                                                 # analytic: one per entry
        want = standin.pool(f, x, p, ALPHAS, const_x=c_x, const_ind=c_i)
        assert _same(phi_a, want[0]) and _same(dphi_a, want[1]) and _same(phi_a, phi)


_REFUSAL = r"""
import ctypes as C, glob, os, subprocess, sys
import numpy as np
root, so = sys.argv[1], sys.argv[2]
host = os.path.join(root, "parallelnonlinearoptimizationlibrary_b200", "host")
subprocess.check_call(["g++", "-std=c++17", "-O2", "-fPIC", "-ffp-contract=off", "-w", "-shared", "-Wl,-Bsymbolic", "-I" + os.path.join(root, "include"),
                       "-I" + host] + sorted(glob.glob(os.path.join(host, "*.cpp"))) +
                      [os.path.join(root, "oracle", "host_logic_device.cpp"), os.path.join(root, "oracle", "pnol_oracle.cpp"), "-o", so])
lib = C.CDLL(so, mode=C.RTLD_LOCAL)
lib.pnolhost_last_error.restype = C.c_char_p
p = lambda a: C.c_void_p(a.ctypes.data)
x, prm = np.full(4, 3.0), np.array([1e-4, 0.9, 1e-6, 1.0, 1000, 1e-7, 1e-3, 5, 1e-5, 1e-5, 0])
f0, fo, it = C.c_double(), C.c_double(), C.c_int()
assert lib.pnolhost_bfgs(b"bfgs", b"rosenbrock", p(x), 4, p(prm), None, None, 0, 0, C.byref(f0), C.byref(fo), C.byref(it)) == 0  # as before
lib.pnolhost_set_analytic_slope(1)
x = np.full(4, 3.0)
st = lib.pnolhost_bfgs(b"bfgs", b"rosenbrock", p(x), 4, p(prm), None, None, 0, 0, C.byref(f0), C.byref(fo), C.byref(it))
print(st, lib.pnolhost_last_error().decode())
"""


def test_analytic_slopes_on_a_c_abi_without_them_are_refused(tmp_path):
    """The host sources reference pnol_alpha_pool_analytic weakly: linked against a C-ABI implementation without it (the unmodified
    stand-in, in a process where no libpnol_b200.so is loaded) they still build and load, and the analytic mode is refused with
    PNOL_ERR_NO_FUNCTOR instead of taking a forward difference."""
    import shutil
    import subprocess
    import sys
    if shutil.which("g++") is None:
        pytest.skip("no g++ on this box")
    r = subprocess.run([sys.executable, "-c", _REFUSAL, UG.ROOT, str(tmp_path / "libstandin.so")], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    st, msg = r.stdout.strip().split(" ", 1)
    assert int(st) == capi.ERR_NO_FUNCTOR and "analytic line-search slopes (Runtime::setAnalyticSlope)" in msg, r.stdout
    assert "not provided by the C-ABI implementation" in msg, r.stdout
