"""Analytic gradients (pnol_gradient) without a GPU: the host side of the one __host__ __device__ partial() per objective
(include/pnol/functors.hpp) against a numpy restatement of its stated operation order (bit for bit) and against a complex-step or
mpmath derivative (to 32 ulp of the gradient's size); sin2pi (include/pnol/pnol_math.h) against mpmath; and the registration rules of
pnol_register_functor_gradient."""
import ctypes as C

import mpmath
import numpy as np
import pytest

import host_logic_gradient_lib as HLG
import user_gradient_lib as UG
from parallelnonlinearoptimizationlibrary_b200 import capi

EPS = 2.0 ** -52


@pytest.fixture(scope="module")
def user():
    return UG.build_and_load()


def test_user_gradient_functors_compile_out_of_tree_and_register(user):
    lib = capi.load_library()
    assert user.my_gradients_registration_status() == 0
    for kind in (UG.MYG_F_TRID, UG.MYG_F_STYBLINSKI):
        assert lib.pnol_functor_registered(kind) == 1 and lib.pnol_functor_has_gradient(kind) == 1
    for kind in (capi.F_ROSENBROCK, capi.F_POWER, capi.F_BOOTH, capi.F_GOLDSTEIN, capi.F_RASTRIGIN, capi.F_EXPCURVE_SINGLE):
        assert lib.pnol_functor_has_gradient(kind) == 1
    for kind in (capi.F_EXPCURVE, capi.F_CUBIC, capi.F_LORENTZ_SUM, 0, 7, capi.F_USER_SCALAR_BASE + 999):
        assert lib.pnol_functor_has_gradient(kind) == 0


# ---- numpy restatements of the header's operation order ----
def np_rosenbrock(x):
    n = x.size
    g = np.empty(n)
    for j in range(n):
        xj = x[j]
        a = 200.0 * (xj - x[j - 1] * x[j - 1]) if j >= 1 else None
        b = -400.0 * xj * (x[j + 1] - xj * xj) - 2.0 * (1 - xj) if j <= n - 2 else None
        g[j] = a + b if (a is not None and b is not None) else (a if a is not None else (b if b is not None else 0.0))
    return g


def np_power(x, p):
    if p <= 0:
        return np.zeros_like(x)
    v = np.ones_like(x)
    for _ in range(p - 1):
        v = v * x
    return float(p) * v


def np_booth(x):
    a = x[0] + 2 * x[1] - 7
    b = 2 * x[0] + x[1] - 5
    return np.array([2 * a + 4 * b, 4 * a + 2 * b] + [0.0] * (x.size - 2))


def np_goldstein(x):
    X, Y = x[0], x[1]
    s = X + Y + 1
    d = 2 * X - 3 * Y
    U = 19 - 14 * X + 3 * (X * X) - 14 * Y + 6 * X * Y + 3 * (Y * Y)
    V = 18 - 32 * X + 12 * (X * X) + 48 * Y - 36 * X * Y + 27 * (Y * Y)
    s2, d2 = s * s, d * d
    A, B = 1 + s2 * U, 30 + d2 * V
    dA = (2 * s) * U + s2 * (-14 + 6 * X + 6 * Y)
    dBx = (4 * d) * V + d2 * (-32 + 24 * X - 36 * Y)
    dBy = (-6 * d) * V + d2 * (48 - 36 * X + 54 * Y)
    return np.array([dA * B + A * dBx, dA * B + A * dBy] + [0.0] * (x.size - 2))


def np_expcurve_single(x, t, y):
    e = UG.host_math("exp", x[1] * t)
    func = x[0] * e + x[2]
    d = y - func
    c = -(d + d)
    terms = (c * e, c * ((x[0] * e) * t), c)
    g = np.zeros(x.size)
    for j in range(3):
        s = 0.0
        for v in terms[j]:
            s = s + v
        g[j] = s
    return g


def _points(rng, n, scale):
    x = rng.uniform(-scale, scale, n)
    x[rng.integers(0, n, max(1, n // 8))] = 0.0
    if n > 3:
        x[1], x[2] = -0.0, 1e-170
    return x


@pytest.mark.parametrize("n", [1, 2, 3, 17, 64])
def test_rosenbrock_and_power_partials_are_the_header_operation_order(user, n):
    rng = np.random.default_rng(n)
    for x in (_points(rng, n, 2.0), _points(rng, n, 1e5), np.ones(n)):
        assert np.array_equal(UG.host_partials(capi.F_ROSENBROCK, x), np_rosenbrock(x))
        for p in (-1, 0, 1, 2, 3, 5):
            assert np.array_equal(UG.host_partials(capi.F_POWER, x, ints=(p,)), np_power(x, p)), p


def test_booth_goldstein_expcurve_partials_are_the_header_operation_order(user):
    rng = np.random.default_rng(7)
    for x in [rng.uniform(-3, 3, 2) for _ in range(50)] + [np.array([0.0, -1.0]), np.array([-0.0, 0.0]), np.array([1e8, -3e7])]:
        assert np.array_equal(UG.host_partials(capi.F_BOOTH, x), np_booth(x))
        assert np.array_equal(UG.host_partials(capi.F_GOLDSTEIN, x), np_goldstein(x))
    x4 = np.array([1.0, 2.0, 0.5, 7.0])          # coordinates past the objective's own give 0
    assert np.array_equal(UG.host_partials(capi.F_BOOTH, x4), np_booth(x4)) and np.array_equal(UG.host_partials(capi.F_GOLDSTEIN, x4), np_goldstein(x4))
    t = np.linspace(-2.0, 3.0, 500)
    y = 1.5 * np.exp(0.7 * t) + 0.2 + 0.01 * rng.normal(size=t.size)
    for x in (np.array([1.3, 0.65, 0.1]), np.array([1.5, 0.7, 0.2]), np.array([-4.0, -1.5, 3.0, 9.0])):
        assert np.array_equal(UG.host_partials(capi.F_EXPCURVE_SINGLE, x, columns=(t, y)), np_expcurve_single(x, t, y))


# ---- sin2pi against mpmath ----
def test_sin2pi_is_within_a_few_1e16_of_mpmath(user):
    rng = np.random.default_rng(2)
    quarters = np.arange(-16, 17) / 4.0
    x = np.concatenate([rng.uniform(-0.5, 0.5, 20000), rng.uniform(-1e6, 1e6, 5000), quarters, quarters + 2.0 ** -40,
                        [0.0, -0.0, 5e-324, -5e-324, 1e-300, 0.25 - 2 ** -54, 0.25 + 2 ** -54, 0.5 - 2 ** -54, 1e15 + 0.25, 2.0 ** 52 - 0.5,
                         2.0 ** 52, 2.0 ** 53 + 2, 1e300, -1e300, 123456789.125, -987654.375]])
    got = UG.host_math("sin2pi", x)
    mpmath.mp.prec = 160
    want = np.array([float(mpmath.sinpi(2 * mpmath.mpf(float(v)))) for v in x])
    err = np.abs(got - want)
    assert err.max() <= 4e-16, (x[np.argmax(err)], err.max())
    exact = {0.0: 0.0, 0.25: 1.0, 0.5: 0.0, 0.75: -1.0, -0.25: -1.0, 1.0: 0.0, 1e300: 0.0, 2.0 ** 52: 0.0}
    for v, w in exact.items():
        assert UG.host_math("sin2pi", np.array([v]))[0] == w, v


# ---- every partial against an independent derivative ----
def cs_gradient(f, x, h=1e-200):
    """complex-step derivative: g[j] = Im f(x + i h e_j) / h"""
    g = np.empty(x.size)
    for j in range(x.size):
        xc = x.astype(np.complex128)
        xc[j] += 1j * h
        g[j] = np.imag(f(xc)) / h
    return g


def assert_within_ulps(g, gref, ulps=32):
    scale = np.maximum(np.abs(gref), np.max(np.abs(gref)))
    bad = np.abs(g - gref) > ulps * EPS * scale
    assert not bad.any(), (np.argwhere(bad)[:5], g[bad][:5], gref[bad][:5])


def test_every_partial_matches_a_complex_step_or_mpmath_derivative(user):
    rng = np.random.default_rng(11)
    x = rng.uniform(-2, 2, 40)
    assert_within_ulps(UG.host_partials(capi.F_ROSENBROCK, x),
                       cs_gradient(lambda z: np.sum(100 * (z[1:] - z[:-1] ** 2) ** 2 + (1 - z[:-1]) ** 2), x))
    for p in (1, 2, 3, 6):
        assert_within_ulps(UG.host_partials(capi.F_POWER, x, ints=(p,)), cs_gradient(lambda z: np.sum(z ** p), x))
    for x2 in (rng.uniform(-3, 3, 2), np.array([1.0, 3.5]), np.array([0.1, -0.9])):       # away from the minima, where g = 0
        assert_within_ulps(UG.host_partials(capi.F_BOOTH, x2),
                           cs_gradient(lambda z: (z[0] + 2 * z[1] - 7) ** 2 + (2 * z[0] + z[1] - 5) ** 2, x2))
        gp = lambda z: ((1 + (z[0] + z[1] + 1) ** 2 * (19 - 14 * z[0] + 3 * z[0] ** 2 - 14 * z[1] + 6 * z[0] * z[1] + 3 * z[1] ** 2)) *  # noqa: E731
                        (30 + (2 * z[0] - 3 * z[1]) ** 2 * (18 - 32 * z[0] + 12 * z[0] ** 2 + 48 * z[1] - 36 * z[0] * z[1] + 27 * z[1] ** 2)))
        assert_within_ulps(UG.host_partials(capi.F_GOLDSTEIN, x2), cs_gradient(gp, x2))
    t = np.linspace(-2.0, 3.0, 300)
    y = 1.5 * np.exp(0.7 * t) + 0.2 + 0.01 * rng.normal(size=t.size)
    x3 = np.array([1.3, 0.65, 0.1])
    assert_within_ulps(UG.host_partials(capi.F_EXPCURVE_SINGLE, x3, columns=(t, y)),
                       cs_gradient(lambda z: np.sum((y - (z[0] * np.exp(z[1] * t) + z[2])) ** 2), x3))
    # Rastrigin: mpmath's derivative of x^2 - 10 cos(2 pi x) at 160 bits
    xr = np.concatenate([rng.uniform(-5.12, 5.12, 300), [0.0, 0.25, 0.5, -1.75, 3.0]])
    mpmath.mp.prec = 160
    want = np.array([float(mpmath.diff(lambda v: v * v - 10 * mpmath.cos(2 * mpmath.pi * v), mpmath.mpf(float(v)))) for v in xr])
    assert_within_ulps(UG.host_partials(capi.F_RASTRIGIN, xr), want)
    # the user's Trid and Styblinski-Tang
    assert_within_ulps(UG.host_partials(UG.MYG_F_TRID, x), cs_gradient(lambda z: np.sum((z - 1) ** 2) - np.sum(z[1:] * z[:-1]), x))
    assert_within_ulps(UG.host_partials(UG.MYG_F_STYBLINSKI, x, scalars=(0.5,)),
                       cs_gradient(lambda z: 0.5 * np.sum(z ** 4 - 16 * z ** 2 + 5 * z), x))


# ---- registration rules (pnol_register_functor_gradient) ----
class VtableV2(C.Structure):
    """pnol_functor_vtable, ABI 2 (include/pnol_b200.h); a version-1 table is the same without the last field"""
    _fields_ = [("abi_version", C.c_int), ("n_columns", C.c_int), ("eval_batch", C.c_void_p), ("fd_points", C.c_void_p),
                ("fd_hessian", C.c_void_p), ("alpha_pool", C.c_void_p), ("residual", C.c_void_p), ("fd_jacobian", C.c_void_p),
                ("jacobian", C.c_void_p)]


def _table(abi, scalar):
    lib = capi.load_library()
    fn = C.cast(lib.pnol_version, C.c_void_p).value        # any non-NULL code address: registration never calls a launcher
    vt = VtableV2()
    vt.abi_version, vt.n_columns = abi, 0
    if scalar:
        vt.eval_batch = vt.fd_points = vt.fd_hessian = vt.alpha_pool = fn
    else:
        vt.residual = vt.fd_jacobian = fn
    return vt


def test_register_functor_gradient_rules():
    lib = capi.load_library()
    fn = C.c_void_p(C.cast(lib.pnol_version, C.c_void_p).value)
    S, R = capi.F_USER_SCALAR_BASE + 700, capi.F_USER_RESIDUAL_BASE + 700
    keep = [_table(1, True), _table(2, True), _table(2, False), _table(2, True)]
    assert lib.pnol_register_functor(S, C.byref(keep[0])) == capi.PNOL_OK          # ABI 1
    assert lib.pnol_register_functor(S + 1, C.byref(keep[1])) == capi.PNOL_OK      # ABI 2
    assert lib.pnol_register_functor(R, C.byref(keep[2])) == capi.PNOL_OK
    for kind in (S, S + 1):
        assert lib.pnol_functor_has_gradient(kind) == 0
        assert lib.pnol_register_functor_gradient(kind, fn) == capi.PNOL_OK
        assert lib.pnol_functor_has_gradient(kind) == 1
    # a residual kind, a kind without a table, a built-in kind, a kind outside every range and NULL are refused
    assert lib.pnol_register_functor_gradient(R, fn) == capi.ERR_INVALID
    assert lib.pnol_register_functor_gradient(S + 2, fn) == capi.ERR_INVALID
    assert lib.pnol_register_functor_gradient(capi.F_ROSENBROCK, fn) == capi.ERR_INVALID
    assert lib.pnol_register_functor_gradient(5000, fn) == capi.ERR_INVALID
    assert lib.pnol_register_functor_gradient(S, None) == capi.ERR_INVALID
    assert lib.pnol_functor_has_gradient(R) == 0 and lib.pnol_functor_has_gradient(S + 2) == 0
    assert lib.pnol_functor_has_gradient(S) == 1                                    # the refused NULL left the launcher in place
    # replacing the table drops the gradient attached to the old one
    assert lib.pnol_register_functor(S, C.byref(keep[3])) == capi.PNOL_OK
    assert lib.pnol_functor_has_gradient(S) == 0 and lib.pnol_functor_registered(S) == 1
    assert lib.pnol_functor_has_gradient(S + 1) == 1


# ---- the host controllers in the analytic mode, without a GPU ----
def _bfgs(lib, variant, obj, x0, params, lb=None, ub=None, pool=0):
    import test_host_logic_cpu as TH
    return TH.bfgs(lib, variant, obj, x0, params, lb, ub, pool)


def test_host_controllers_take_the_partials_in_the_analytic_mode(user):
    """The unmodified host sources on the CPU stand-in extended by the host partials (tests/host_logic_gradient.cpp):
    Objective::gradientApproximation[MPI][Recur] return partial()'s bits and ignore dX, and BFGS / BFGS_Bnd_MPI_SW reach the optima."""
    hl = HLG.build_and_load()
    if hl is None:
        pytest.skip("no g++ on this box")
    p = lambda a: C.c_void_p(a.ctypes.data)                         # noqa: E731
    hl.pnolhost_set_analytic_gradient(1)
    try:
        for obj, kind, n in (("rosenbrock", capi.F_ROSENBROCK, 40), ("booth", capi.F_BOOTH, 2), ("goldstein", capi.F_GOLDSTEIN, 2),
                             ("rastrigin", capi.F_RASTRIGIN, 12), ("power:3", capi.F_POWER, 5)):
            x = np.random.default_rng(n).uniform(-1.5, 1.5, n)
            want = UG.host_partials(kind, x, ints=(3,) if kind == capi.F_POWER else ())
            for which in (0, 1):
                g = np.empty(n)
                assert hl.pnolhost_gradient(obj.encode(), p(x), p(np.full(n, np.nan)), n, which, p(g)) == 0, hl.pnolhost_last_error()
                assert np.array_equal(g, want), (obj, which)
            ind = np.zeros(n, np.uint8)
            ind[::3] = 1
            xr = np.ascontiguousarray(x[ind == 0])
            gr, f = np.empty(xr.size), C.c_double()
            assert hl.pnolhost_gradient_recur(obj.encode(), p(xr), p(np.full(xr.size, 1e-7)), xr.size, p(x), p(ind), n, p(gr), C.byref(f)) == 0
            assert np.array_equal(gr, want[ind == 0]), obj
        BF = [1e-4, 0.9, 1e-6, 1.0, 1000, 1e-7, 1e-3, 1000, 1e-5, 1e-5, 0]
        SW = [1e-4, 0.8, 1e-6, 1.0, 1e-10, 2.0, 50, 1e-5, 1e-6, 1e-3, 1000, 1e-5, 1e-5, 0]
        for obj, x0, xopt in (("rosenbrock", np.full(10, 3.0), np.ones(10)), ("booth", np.array([3.0, -2.0]), np.array([1.0, 3.0]))):
            for r in (_bfgs(hl, "bfgs", obj, x0, BF), _bfgs(hl, "bfgs_bnd_sw", obj, x0, SW, np.full(x0.size, -5.0), np.full(x0.size, 5.0), 8)):
                assert np.linalg.norm(r["X"] - xopt) <= 1e-4 * np.linalg.norm(xopt) and r["fOpt"] < 1e-8, (obj, r)
    finally:
        hl.pnolhost_set_analytic_gradient(0)


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
x, dx, g = np.full(4, 0.5), np.full(4, 1e-7), np.empty(4)
p = lambda a: C.c_void_p(a.ctypes.data)
assert lib.pnolhost_gradient(b"rosenbrock", p(x), p(dx), 4, 0, p(g)) == 0        # the forward difference works as before
lib.pnolhost_set_analytic_gradient(1)
st = lib.pnolhost_gradient(b"rosenbrock", p(x), p(dx), 4, 0, p(g))
print(st, lib.pnolhost_last_error().decode())
"""


def test_analytic_mode_on_a_c_abi_without_the_gradient_is_refused(tmp_path):
    """The host sources reference pnol_gradient[_recur] weakly: linked against a C-ABI implementation without them (the unmodified
    stand-in, in a process where no libpnol_b200.so is loaded) they still build and load, and the analytic mode is refused with
    PNOL_ERR_NO_FUNCTOR instead of computing anything."""
    import shutil
    import subprocess
    import sys
    if shutil.which("g++") is None:
        pytest.skip("no g++ on this box")
    r = subprocess.run([sys.executable, "-c", _REFUSAL, UG.ROOT, str(tmp_path / "libstandin.so")], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    st, msg = r.stdout.strip().split(" ", 1)
    assert int(st) == capi.ERR_NO_FUNCTOR and "not provided by the C-ABI implementation" in msg, r.stdout
