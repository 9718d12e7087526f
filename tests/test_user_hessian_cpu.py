"""Analytic Hessians (pnol_hessian) without a GPU: the host side of the one __host__ __device__ partial2() per objective
(include/pnol/functors.hpp, the user's tests/user_functor/my_hessians.hpp) against a numpy restatement of its stated operation order
(bit for bit) and against a complex-step derivative of the gradient or an mpmath second derivative (to 32 ulp of the Hessian's largest
entry); the registration rules of pnol_register_functor_hessian; and the BFGS controllers with initHessFD in the analytic mode on the CPU
stand-in extended by the host partial2() (tests/host_logic_standin.cpp)."""
import ctypes as C

import mpmath
import numpy as np
import pytest

import host_standin
import user_gradient_lib as UG
import user_hessian_lib as UH
from parallelnonlinearoptimizationlibrary_b200 import capi

EPS = 2.0 ** -52
SCALAR_BUILTINS = (capi.F_ROSENBROCK, capi.F_POWER, capi.F_BOOTH, capi.F_GOLDSTEIN, capi.F_RASTRIGIN, capi.F_EXPCURVE_SINGLE)


@pytest.fixture(scope="module")
def user():
    return UH.build_and_load()


def test_user_hessian_functors_compile_out_of_tree_and_register(user):
    lib = capi.load_library()
    assert user.my_hessians_registration_status() == 0
    for kind in (UH.MYH_F_QUADFORM, UH.MYH_F_STYBLINSKI):
        assert lib.pnol_functor_registered(kind) == 1 and lib.pnol_functor_has_hessian(kind) == 1
        assert lib.pnol_functor_has_gradient(kind) == 0                  # partial2() without partial()
    for kind in SCALAR_BUILTINS:
        assert lib.pnol_functor_has_hessian(kind) == 1
    UG.build_and_load()
    assert lib.pnol_functor_has_gradient(UG.MYG_F_TRID) == 1 and lib.pnol_functor_has_hessian(UG.MYG_F_TRID) == 0  # partial() only
    for kind in (capi.F_EXPCURVE, capi.F_CUBIC, capi.F_LORENTZ_SUM, 0, 7, capi.F_USER_SCALAR_BASE + 999):
        assert lib.pnol_functor_has_hessian(kind) == 0


# ---- numpy restatements of the header's operation order (upper triangle, mirrored) ----
def _mirror(H):
    iu = np.triu_indices(H.shape[0], 1)
    H[(iu[1], iu[0])] = H[iu]
    return H


def np_rosenbrock(x):
    n = x.size
    H = np.zeros((n, n))
    for j in range(n):
        b = 1200.0 * (x[j] * x[j]) - 400.0 * x[j + 1] + 2.0 if j <= n - 2 else None
        if j >= 1 and b is not None:
            H[j, j] = 200.0 + b
        elif j >= 1:
            H[j, j] = 200.0
        elif b is not None:
            H[j, j] = b
        if j <= n - 2:
            H[j, j + 1] = -400.0 * x[j]
    return _mirror(H)


def np_power(x, p):
    H = np.zeros((x.size, x.size))
    if p > 1:
        v = np.ones_like(x)
        for _ in range(p - 2):
            v = v * x
        H[np.diag_indices(x.size)] = float(p * (p - 1)) * v
    return H


def np_booth(x):
    H = np.zeros((x.size, x.size))
    H[:2, :2] = [[10.0, 8.0], [8.0, 10.0]]
    return H


def np_goldstein(x):
    X, Y = x[0], x[1]
    s = X + Y + 1
    d = 2 * X - 3 * Y
    U = 19 - 14 * X + 3 * (X * X) - 14 * Y + 6 * X * Y + 3 * (Y * Y)
    V = 18 - 32 * X + 12 * (X * X) + 48 * Y - 36 * X * Y + 27 * (Y * Y)
    s2, d2 = s * s, d * d
    A, B = 1 + s2 * U, 30 + d2 * V
    Ux = -14 + 6 * X + 6 * Y
    Vx, Vy = -32 + 24 * X - 36 * Y, 48 - 36 * X + 54 * Y
    dA = (2 * s) * U + s2 * Ux
    Bd = ((4 * d) * V + d2 * Vx, (-6 * d) * V + d2 * Vy)
    A2 = 2 * U + (4 * s) * Ux + 6 * s2
    B2 = {(0, 0): 8 * V + (8 * d) * Vx + 24 * d2, (0, 1): -12 * V + (4 * d) * Vy - (6 * d) * Vx - 36 * d2,
          (1, 1): 18 * V - (12 * d) * Vy + 54 * d2}
    H = np.zeros((x.size, x.size))
    for (i, j), b2 in B2.items():
        H[i, j] = A2 * B + dA * Bd[j] + dA * Bd[i] + A * b2
    return _mirror(H)


def np_rastrigin(x):
    return np.diag(2 + 394.78417604357435 * UG.host_math("cos2pi", x))


def np_expcurve_single(x, t, y):
    e = UG.host_math("exp", x[1] * t)
    func = x[0] * e + x[2]
    d = y - func
    g1 = (x[0] * e) * t
    g = (e, g1, np.ones_like(t))
    h = {(0, 1): e * t, (1, 1): g1 * t}
    H = np.zeros((x.size, x.size))
    for i in range(3):
        for j in range(i, 3):
            terms = 2.0 * (g[i] * g[j]) - (2.0 * d) * h.get((i, j), np.zeros_like(t))
            s = 0.0
            for v in terms:
                s = s + v
            H[i, j] = s
    return _mirror(H)


def np_quadform(x, A):
    n = x.size
    M = A.reshape(n, n)
    return _mirror(np.triu(0.5 * (M + M.T)))


def np_styblinski(x, s):
    return np.diag(s * (12.0 * (x * x) - 32.0))


def _points(rng, n, scale):
    x = rng.uniform(-scale, scale, n)
    x[rng.integers(0, n, max(1, n // 8))] = 0.0
    if n > 3:
        x[1], x[2] = -0.0, 1e-170
    return x


def _same(a, b):
    """bit for bit, +0 and -0 told apart"""
    return a.shape == b.shape and np.array_equal(a.view(np.int64), b.view(np.int64))


@pytest.mark.parametrize("n", [1, 2, 3, 17, 64])
def test_separable_and_banded_hessians_are_the_header_operation_order(user, n):
    rng = np.random.default_rng(n)
    for x in (_points(rng, n, 2.0), _points(rng, n, 1e5), np.ones(n)):
        assert _same(UH.host_hessian(capi.F_ROSENBROCK, x), np_rosenbrock(x))
        for p in (-1, 0, 1, 2, 3, 5):
            assert _same(UH.host_hessian(capi.F_POWER, x, ints=(p,)), np_power(x, p)), p
        assert _same(UH.host_hessian(capi.F_RASTRIGIN, x), np_rastrigin(x))
        assert _same(UH.host_hessian(UH.MYH_F_STYBLINSKI, x, scalars=(0.5,)), np_styblinski(x, 0.5))
        A = rng.normal(size=n * n)
        assert _same(UH.host_hessian(UH.MYH_F_QUADFORM, x, columns=(A,)), np_quadform(x, A))


def test_booth_goldstein_expcurve_hessians_are_the_header_operation_order(user):
    rng = np.random.default_rng(7)
    for x in [rng.uniform(-3, 3, 2) for _ in range(50)] + [np.array([0.0, -1.0]), np.array([-0.0, 0.0]), np.array([1e8, -3e7])]:
        assert _same(UH.host_hessian(capi.F_BOOTH, x), np_booth(x))
        assert _same(UH.host_hessian(capi.F_GOLDSTEIN, x), np_goldstein(x))
    x4 = np.array([1.0, 2.0, 0.5, 7.0])          # coordinates past the objective's own give 0
    assert _same(UH.host_hessian(capi.F_BOOTH, x4), np_booth(x4)) and _same(UH.host_hessian(capi.F_GOLDSTEIN, x4), np_goldstein(x4))
    t = np.linspace(-2.0, 3.0, 500)
    y = 1.5 * np.exp(0.7 * t) + 0.2 + 0.01 * rng.normal(size=t.size)
    for x in (np.array([1.3, 0.65, 0.1]), np.array([1.5, 0.7, 0.2]), np.array([-4.0, -1.5, 3.0, 9.0])):
        assert _same(UH.host_hessian(capi.F_EXPCURVE_SINGLE, x, columns=(t, y)), np_expcurve_single(x, t, y))


def test_pairs_entry_point_is_the_whole_matrix_entry_point(user):
    rng = np.random.default_rng(3)
    x = rng.uniform(-2, 2, 40)
    ii, jj = np.triu_indices(40)
    assert _same(UH.host_partial2(capi.F_ROSENBROCK, x, ii, jj), UH.host_hessian(capi.F_ROSENBROCK, x)[ii, jj])


# ---- every Hessian against an independent derivative ----
def cs_hessian(grad, x, h=1e-200):
    """complex-step derivative of a complex-safe gradient: H[:, j] = Im grad(x + i h e_j) / h"""
    H = np.empty((x.size, x.size))
    for j in range(x.size):
        xc = x.astype(np.complex128)
        xc[j] += 1j * h
        H[:, j] = np.imag(grad(xc)) / h
    return H


def assert_within_ulps(H, Href, ulps=32):
    scale = np.max(np.abs(Href))
    bad = np.abs(H - Href) > ulps * EPS * scale
    assert not bad.any(), (np.argwhere(bad)[:5], H[bad][:5], Href[bad][:5])


def g_rosenbrock(z):
    g = np.zeros(z.size, dtype=z.dtype)
    g[1:] += 200 * (z[1:] - z[:-1] ** 2)
    g[:-1] += -400 * z[:-1] * (z[1:] - z[:-1] ** 2) - 2 * (1 - z[:-1])
    return g


def g_goldstein(z):
    X, Y = z[0], z[1]
    s, d = X + Y + 1, 2 * X - 3 * Y
    U = 19 - 14 * X + 3 * X * X - 14 * Y + 6 * X * Y + 3 * Y * Y
    V = 18 - 32 * X + 12 * X * X + 48 * Y - 36 * X * Y + 27 * Y * Y
    A, B = 1 + s * s * U, 30 + d * d * V
    dA = 2 * s * U + s * s * (-14 + 6 * X + 6 * Y)
    dBx = 4 * d * V + d * d * (-32 + 24 * X - 36 * Y)
    dBy = -6 * d * V + d * d * (48 - 36 * X + 54 * Y)
    return np.array([dA * B + A * dBx, dA * B + A * dBy])


def test_every_hessian_matches_a_complex_step_or_mpmath_derivative(user):
    rng = np.random.default_rng(11)
    x = rng.uniform(-2, 2, 40)
    assert_within_ulps(UH.host_hessian(capi.F_ROSENBROCK, x), cs_hessian(g_rosenbrock, x))
    for p in (1, 2, 3, 6):
        assert_within_ulps(UH.host_hessian(capi.F_POWER, x, ints=(p,)), cs_hessian(lambda z: p * z ** (p - 1), x))
    for x2 in (rng.uniform(-3, 3, 2), np.array([1.0, 3.5]), np.array([0.1, -0.9]), np.array([0.0, -1.0])):
        assert_within_ulps(UH.host_hessian(capi.F_BOOTH, x2),
                           cs_hessian(lambda z: np.array([2 * (z[0] + 2 * z[1] - 7) + 4 * (2 * z[0] + z[1] - 5),
                                                          4 * (z[0] + 2 * z[1] - 7) + 2 * (2 * z[0] + z[1] - 5)]), x2))
        assert_within_ulps(UH.host_hessian(capi.F_GOLDSTEIN, x2), cs_hessian(g_goldstein, x2))
    t = np.linspace(-2.0, 3.0, 300)
    y = 1.5 * np.exp(0.7 * t) + 0.2 + 0.01 * rng.normal(size=t.size)

    def g_exp(z):
        e = np.exp(z[1] * t)
        c = -2 * (y - (z[0] * e + z[2]))
        return np.array([np.sum(c * e), np.sum(c * z[0] * e * t), np.sum(c)])
    x3 = np.array([1.3, 0.65, 0.1])
    assert_within_ulps(UH.host_hessian(capi.F_EXPCURVE_SINGLE, x3, columns=(t, y)), cs_hessian(g_exp, x3))
    # Rastrigin: mpmath's second derivative of x^2 - 10 cos(2 pi x) at 160 bits, against the largest diagonal entry
    xr = np.concatenate([rng.uniform(-5.12, 5.12, 300), [0.0, 0.25, 0.5, -1.75, 3.0]])
    mpmath.mp.prec = 160
    want = np.array([float(mpmath.diff(lambda v: v * v - 10 * mpmath.cos(2 * mpmath.pi * v), mpmath.mpf(float(v)), 2)) for v in xr])
    got = np.diag(UH.host_hessian(capi.F_RASTRIGIN, xr))
    assert np.max(np.abs(got - want)) <= 32 * EPS * np.max(np.abs(want)), np.max(np.abs(got - want))
    # the user's quadratic form and Styblinski-Tang
    A = rng.normal(size=40 * 40)
    M = A.reshape(40, 40)
    assert_within_ulps(UH.host_hessian(UH.MYH_F_QUADFORM, x, columns=(A,)), cs_hessian(lambda z: 0.5 * (M + M.T) @ z, x))
    assert_within_ulps(UH.host_hessian(UH.MYH_F_STYBLINSKI, x, scalars=(0.5,)), cs_hessian(lambda z: 0.5 * (4 * z ** 3 - 32 * z + 5), x))


# ---- registration rules (pnol_register_functor_hessian) ----
def test_register_functor_hessian_rules():
    from test_user_gradient_cpu import _table
    lib = capi.load_library()
    fn = C.c_void_p(C.cast(lib.pnol_version, C.c_void_p).value)      # any non-NULL code address: registration never calls a launcher
    S, R = capi.F_USER_SCALAR_BASE + 710, capi.F_USER_RESIDUAL_BASE + 710
    keep = [_table(1, True), _table(2, True), _table(2, False), _table(2, True)]
    assert lib.pnol_register_functor(S, C.byref(keep[0])) == capi.PNOL_OK          # ABI 1
    assert lib.pnol_register_functor(S + 1, C.byref(keep[1])) == capi.PNOL_OK      # ABI 2
    assert lib.pnol_register_functor(R, C.byref(keep[2])) == capi.PNOL_OK
    for kind in (S, S + 1):
        assert lib.pnol_functor_has_hessian(kind) == 0
        assert lib.pnol_register_functor_hessian(kind, fn) == capi.PNOL_OK
        assert lib.pnol_functor_has_hessian(kind) == 1
        assert lib.pnol_functor_has_gradient(kind) == 0                            # the two derivatives are attached separately
    assert lib.pnol_register_functor_gradient(S, fn) == capi.PNOL_OK
    # a residual kind, a kind without a table, a built-in kind, a kind outside every range and NULL are refused
    assert lib.pnol_register_functor_hessian(R, fn) == capi.ERR_INVALID
    assert lib.pnol_register_functor_hessian(S + 2, fn) == capi.ERR_INVALID
    assert lib.pnol_register_functor_hessian(capi.F_ROSENBROCK, fn) == capi.ERR_INVALID
    assert lib.pnol_register_functor_hessian(5000, fn) == capi.ERR_INVALID
    assert lib.pnol_register_functor_hessian(S, None) == capi.ERR_INVALID
    assert lib.pnol_functor_has_hessian(R) == 0 and lib.pnol_functor_has_hessian(S + 2) == 0
    assert lib.pnol_functor_has_hessian(S) == 1                                     # the refused NULL left the launcher in place
    # replacing the table drops the Hessian (and the gradient) attached to the old one
    assert lib.pnol_register_functor(S, C.byref(keep[3])) == capi.PNOL_OK
    assert lib.pnol_functor_has_hessian(S) == 0 and lib.pnol_functor_has_gradient(S) == 0 and lib.pnol_functor_registered(S) == 1
    assert lib.pnol_functor_has_hessian(S + 1) == 1


# ---- the host controllers in the analytic mode, without a GPU ----
def bfgs_params(variant, iters, inithess=1):
    """setParams of the five BFGS classes (host_capi.cpp: pnolhost_bfgs), the examples' settings"""
    if variant == "bfgs":
        return [1e-4, 0.9, 1e-6, 1.0, 1000, 1e-7, 1e-3, iters, 1e-5, 1e-5, inithess]
    if variant == "bfgs_mpi":
        return [1e-4, 0.9, 4.0, 1.0, 50, 1e-7, 1e-3, iters, 1e-5, 1e-5, inithess]
    if variant == "bfgsbnd_mpi":
        return [1e-4, 0.1, 1e-16, 4.0, 1.0, 1000, 1e-7, 1e-3, iters, 1e-5, 1e-5, 1e-5, inithess]
    return [1e-4, 0.8, 1e-6, 1.0, 1e-10, 2.0, 50, 1e-5, 1e-6, 1e-3, iters, 1e-5, 1e-5, inithess]      # bfgs_bnd, bfgs_bnd_sw


VARIANTS = {"bfgs": 0, "bfgs_mpi": 4, "bfgs_bnd": 0, "bfgs_bnd_sw": 8, "bfgsbnd_mpi": 4}        # variant: pool width
PROBLEMS = [("rosenbrock", np.full(10, 3.0), np.ones(10), 0.0), ("booth", np.array([3.0, -2.0]), np.array([1.0, 3.0]), 0.0),
            ("goldstein", np.array([0.1, -0.9]), np.array([0.0, -1.0]), 3.0)]


def run_bfgs(call, variant, obj, x0, iters):
    """call(variant, obj, x0, params, lb, ub, pool) -> result dict; bounded variants get the box [-5, 5]"""
    bounded = variant in ("bfgs_bnd", "bfgs_bnd_sw", "bfgsbnd_mpi")
    lb, ub = (np.full(x0.size, -5.0), np.full(x0.size, 5.0)) if bounded else (None, None)
    return call(variant, obj, x0, bfgs_params(variant, iters), lb, ub, VARIANTS[variant])


def test_host_hessian_member_takes_partial2_in_the_analytic_mode(user):
    """Objective::hessianApproximation on the stand-in extended by the host partial2(): partial2()'s bits, dX ignored; the forward
    difference when the switch is off."""
    hl = host_standin.load()
    if hl is None:
        pytest.skip("no g++ on this box")
    p = lambda a: C.c_void_p(a.ctypes.data)                         # noqa: E731
    for obj, kind, n in (("rosenbrock", capi.F_ROSENBROCK, 12), ("booth", capi.F_BOOTH, 2), ("goldstein", capi.F_GOLDSTEIN, 2),
                         ("rastrigin", capi.F_RASTRIGIN, 7), ("power:3", capi.F_POWER, 5)):
        x = np.random.default_rng(n).uniform(-1.5, 1.5, n)
        want = UH.host_hessian(kind, x, ints=(3,) if kind == capi.F_POWER else ())
        H = np.empty((n, n))
        hl.pnolhost_set_analytic_hessian(1)
        try:
            assert hl.pnolhost_hessian(obj.encode(), p(x), p(np.full(n, np.nan)), n, p(H)) == 0, hl.pnolhost_last_error()
        finally:
            hl.pnolhost_set_analytic_hessian(0)
        assert _same(H, want), obj
        assert hl.pnolhost_hessian(obj.encode(), p(x), p(np.full(n, 1e-4)), n, p(H)) == 0
        assert not _same(H, want) and np.all(np.isfinite(H)), obj


@pytest.mark.parametrize("variant", sorted(VARIANTS))
def test_bfgs_controllers_start_from_the_analytic_hessian(user, variant):
    """initHessFD = 1 with analytic gradient and Hessian: the five BFGS classes on the extended stand-in reach the known optima."""
    import test_host_logic_cpu as TH
    hl = host_standin.load()
    if hl is None:
        pytest.skip("no g++ on this box")
    hl.pnolhost_set_analytic_gradient(1)
    hl.pnolhost_set_analytic_hessian(1)
    try:
        for obj, x0, xopt, fopt in PROBLEMS:
            if obj == "rosenbrock" and variant in ("bfgs_mpi", "bfgsbnd_mpi"):
                continue            # these two stop short of the optimum from this start with the forward-difference Hessian too
            r = run_bfgs(lambda v, o, x, p, lb, ub, pool: TH.bfgs(hl, v, o, x, p, lb, ub, pool), variant, obj, x0, 1000)
            assert np.linalg.norm(r["X"] - xopt) <= 1e-4 * max(np.linalg.norm(xopt), 1.0), (obj, r)
            assert abs(r["fOpt"] - fopt) < 1e-8, (obj, r)
    finally:
        hl.pnolhost_set_analytic_gradient(0)
        hl.pnolhost_set_analytic_hessian(0)


_REFUSAL = r"""
import ctypes as C, sys
import numpy as np
lib = C.CDLL(sys.argv[1], mode=C.RTLD_LOCAL)
lib.pnolhost_last_error.restype = C.c_char_p
x, dx, H = np.full(4, 0.5), np.full(4, 1e-4), np.empty(16)
p = lambda a: C.c_void_p(a.ctypes.data)
assert lib.pnolhost_hessian(b"rosenbrock", p(x), p(dx), 4, p(H)) == 0        # the forward difference works as before
lib.pnolhost_set_analytic_hessian(1)
st = lib.pnolhost_hessian(b"rosenbrock", p(x), p(dx), 4, p(H))
print(st, lib.pnolhost_last_error().decode())
"""


def test_analytic_hessian_on_a_c_abi_without_it_is_refused():
    """The host sources reference pnol_hessian weakly: linked against a C-ABI implementation without it (the unmodified stand-in, in a
    process where no libpnol_b200.so is loaded) they still build and load, and the analytic mode is refused with PNOL_ERR_NO_FUNCTOR
    instead of computing anything."""
    import subprocess
    import sys
    so = host_standin.base_path()
    if so is None:
        pytest.skip("no g++ on this box")
    r = subprocess.run([sys.executable, "-c", _REFUSAL, so], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    st, msg = r.stdout.strip().split(" ", 1)
    assert int(st) == capi.ERR_NO_FUNCTOR and "analytic Hessians (Runtime::setAnalyticHessian)" in msg, r.stdout
    assert "not provided by the C-ABI implementation" in msg, r.stdout
