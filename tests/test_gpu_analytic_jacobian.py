"""GPU: analytic Jacobians (PNOL_JAC_ANALYTIC). The kernels return the bits of the models' one __host__ __device__ definition
(include/pnol/functors.hpp: R::jacobian, lorentz_term_grad) run on the host: the sum-of-Lorentzians kernel and the generic template
(include/pnol/device/functor_kernels.cuh) for the built-in and the user's models (tests/user_functor/my_jacobians.*). The fused
J^T F, the LM step and the device-resident LM loop with analytic derivatives, and the refusals of models that have none."""
import ctypes as C
import math

import numpy as np
import pytest
import scipy.linalg

import user_jacobian_lib as UJ
from parallelnonlinearoptimizationlibrary_b200 import capi, problems

pytestmark = pytest.mark.gpu

AN = capi.JAC_ANALYTIC
U = 2.0 ** -53


@pytest.fixture(scope="module")
def user():
    return UJ.build_and_load()


def lorentz(ctx, pr, kind=capi.F_LORENTZ_SUM):
    return ctx.functor(kind, (pr["w"],), (), (pr["t"], pr["y"]), pr["m"])


def np_lorentz_grad(a, c, w, t):
    """lorentz_term_grad in the header's operation order"""
    d = t[:, None] - c[None, :]
    u = 1.0 / (1.0 + w * (d * d))
    J = np.empty((t.size, 2 * a.size))
    J[:, 0::2], J[:, 1::2] = -u, -((a[None, :] * u) * u * ((w + w) * d))
    return J


def two_product_sum(J, F):
    """error-free J^T F: math.fsum over the exact two-products (Veltkamp split) of every column"""
    def split(a):
        c = 134217729.0 * a
        hi = c - (c - a)
        return hi, a - hi
    fh, fl = split(F)
    out = np.empty(J.shape[1])
    for j in range(J.shape[1]):
        a = J[:, j]
        p = a * F
        ah, al = split(a)
        e = ((ah * fh - p) + ah * fl + al * fh) + al * fl
        out[j] = math.fsum(np.concatenate([p, e]))
    return out


def assert_jtf_bound(got, J, F):
    m = J.shape[0]
    gamma = m * U / (1.0 - m * U)
    exact = two_product_sum(J, F)
    bound = gamma * (np.abs(J).T @ np.abs(F))
    assert np.all(np.abs(got - exact) <= bound), np.max(np.abs(got - exact) / np.maximum(bound, 1e-300))


# ---------------------------------------------------------------------------------------------------------------------------------
# J bit for bit against the host definition
# ---------------------------------------------------------------------------------------------------------------------------------
def _case(name):
    rng = np.random.default_rng(len(name))
    if name == "expcurve":
        t = np.linspace(-2.0, 3.0, 5003)
        return capi.F_EXPCURVE, (), (t, 1.5 * np.exp(0.7 * t) + 0.2 + 0.01 * rng.normal(size=t.size)), np.array([1.3, 0.65, 0.1])
    if name == "cubic":
        xs = rng.uniform(-3.0, 3.0, 3001)
        return capi.F_CUBIC, (), (xs ** 3, xs, rng.normal(size=xs.size)), np.array([0.5, -1.0, 2.0, 0.25])
    if name in ("lorentz", "user_lorentz"):
        pr = problems.lorentz_problem(10_007, 16)
        return (capi.F_LORENTZ_SUM if name == "lorentz" else UJ.MYJ_F_LORENTZ), (pr["w"],), (pr["t"], pr["y"]), pr["x0"]
    t = np.linspace(-3.0, 5.0, 2001)
    return UJ.MYJ_F_GAUSS, (0.3,), (t, 2.5 * np.exp(-(t - 1.2) ** 2 * 0.8) + 0.3), np.array([2.2, 1.05, 0.9])


@pytest.mark.parametrize("name", ["expcurve", "cubic", "lorentz", "user_lorentz", "user_gauss"])
def test_analytic_jacobian_equals_the_host_definition(ctx, user, name):
    kind, scalars, cols, x = _case(name)
    f = ctx.functor(kind, scalars, (), cols, cols[0].size)
    J, F = ctx.fd_jacobian(f, x, None, mode=AN)
    Jh, Fh = UJ.host_jacobian(kind, scalars, cols, x)
    assert np.array_equal(J, Jh) and np.array_equal(F, Fh)
    assert np.array_equal(F, ctx.residual_eval(f, x)[0])          # F has the bits of pnol_residual_eval


@pytest.mark.parametrize("K,m", [(K, m) for K in (1, 2, 8, 32, 128, 256) for m in (1, 7, 9, 255, 257, 5003)] +
                         [(512, 33), (1024, 17), (4096, 9)])
def test_lorentz_kernel_writes_every_entry(ctx, user, K, m):
    pr = problems.lorentz_problem(m, K)
    n = pr["n"]
    f = lorentz(ctx, pr)
    Jd = ctx.to_device(np.full(m * n, np.nan))
    Fd = ctx.to_device(np.full(m, np.nan))
    try:
        ctx.fd_jacobian(f, pr["x0"], None, J=Jd, F=Fd, mode=AN, n=n)
        J, F = ctx.to_host(Jd, (m, n)), ctx.to_host(Fd, m)
    finally:
        ctx.free(Jd)
        ctx.free(Fd)
    Jh, Fh = UJ.host_jacobian(capi.F_LORENTZ_SUM, (pr["w"],), (pr["t"], pr["y"]), pr["x0"])
    assert np.array_equal(J, Jh) and np.array_equal(F, Fh)
    assert np.array_equal(J, np_lorentz_grad(pr["x0"][0::2], pr["x0"][1::2], pr["w"], pr["t"]))


def test_lorentz_kernel_at_the_benchmark_shape(ctx, user):
    m, K = 4_000_000, 128
    pr = problems.lorentz_problem(m, K)
    n = pr["n"]
    f = lorentz(ctx, pr)
    rows = np.unique(np.concatenate([[0, 1, m - 2, m - 1], np.random.default_rng(1).integers(0, m, 200)]))
    Jd = ctx.malloc(m * n * 8)
    try:
        ctx.fd_jacobian(f, pr["x0"], None, J=Jd, mode=AN, n=n)
        got = np.stack([ctx.to_host(Jd + int(i) * n * 8, n) for i in rows])
    finally:
        ctx.free(Jd)
    Jh, _ = UJ.host_jacobian(capi.F_LORENTZ_SUM, (pr["w"],), (pr["t"], pr["y"]), pr["x0"], rows=rows)
    assert np.array_equal(got, Jh)


@pytest.mark.parametrize("K,m", [(8, 3001), (128, 2049)])
def test_misaligned_j_and_the_user_copy_give_the_same_bits(ctx, user, K, m):
    """J offset by one double: the 16-byte stores of the Lorentz kernel cannot take it, the generic template does; and the user's
    copy of the model through the generic template equals the built-in kernel"""
    pr = problems.lorentz_problem(m, K)
    n = pr["n"]
    J, F = ctx.fd_jacobian(lorentz(ctx, pr), pr["x0"], None, mode=AN)
    base = ctx.to_device(np.full(m * n + 2, np.nan))
    try:
        ctx.fd_jacobian(lorentz(ctx, pr), pr["x0"], None, J=base + 8, mode=AN, n=n)
        Jmis = ctx.to_host(base + 8, (m, n))
    finally:
        ctx.free(base)
    assert np.array_equal(Jmis, J)
    Ju, Fu = ctx.fd_jacobian(lorentz(ctx, pr, UJ.MYJ_F_LORENTZ), pr["x0"], None, mode=AN)
    assert np.array_equal(Ju, J) and np.array_equal(Fu, F)


# ---------------------------------------------------------------------------------------------------------------------------------
# fused J^T F and the normal equations of the LM step
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K,m", [(8, 100_000), (128, 50_000)])
def test_fused_jtf_of_a_one_hot_residual_is_the_row_of_j(ctx, user, K, m):
    pr = problems.lorentz_problem(m, K)
    n = pr["n"]
    f = lorentz(ctx, pr)
    Jd, Fd, Ft, JTJd = ctx.malloc(m * n * 8), ctx.malloc(m * 8), ctx.malloc(m * 8), ctx.malloc((n * n + n) * 8)
    try:
        for i in (0, 77, m // 3, m // 2 + 5, m - 1):            # rows of different blocks, the last one included
            e = np.zeros(m)
            e[i] = 1.0
            ctx.memcpy(Fd, e, m * 8)
            ctx.lm_step(f, pr["x0"], None, n, Jd, Fd, Ft, 1e-3, JTJd, jac_mode=AN)
            jtf = -ctx.to_host(JTJd + n * n * 8, n)
            assert np.array_equal(jtf, ctx.to_host(Jd + i * n * 8, n)), i
    finally:
        for p in (Jd, Fd, Ft, JTJd):
            ctx.free(p)


@pytest.mark.parametrize("K,m", [(8, 100_000), (128, 60_000)])
def test_step_normal_equations_with_a_real_residual(ctx, user, K, m):
    pr = problems.lorentz_problem(m, K)
    n = pr["n"]
    f = lorentz(ctx, pr)
    Jd, Fd, Ft, JTJd = ctx.malloc(m * n * 8), ctx.malloc(m * 8), ctx.malloc(m * 8), ctx.malloc((n * n + n) * 8)
    try:
        F, _ = ctx.residual_eval(f, pr["x0"], F=Fd, n=n)
        F = ctx.to_host(Fd, m)
        ctx.lm_step(f, pr["x0"], None, n, Jd, Fd, Ft, 1e-3, JTJd, jac_mode=AN)
        J = ctx.to_host(Jd, (m, n))
        step = ctx.to_host(JTJd, n * n + n)
        JTJ_ne, _, _ = ctx.lm_normal_eq(Jd, None, m, n, 1e-3)
        _, _, rhs_ne = ctx.lm_normal_eq(Jd, Fd, m, n, 1e-3)
    finally:
        for p in (Jd, Fd, Ft, JTJd):
            ctx.free(p)
    assert np.array_equal(J, np_lorentz_grad(pr["x0"][0::2], pr["x0"][1::2], pr["w"], pr["t"]))
    assert np.array_equal(step[:n * n].reshape(n, n), JTJ_ne)     # J^T J of the step = pnol_lm_normal_eq on the same J
    assert_jtf_bound(-step[n * n:], J, F)                          # J^T F summed by the Jacobian kernel
    assert_jtf_bound(-rhs_ne, J, F)                                # ... and by the SYRK


def test_row_blocked_step_equals_the_stored_j_step(ctx, user, monkeypatch):
    m, K = 30_000, 16
    pr = problems.lorentz_problem(m, K)
    n = pr["n"]
    f = lorentz(ctx, pr)
    Jd, Fd, Ft, JTJd = ctx.malloc(m * n * 8), ctx.malloc(m * 8), ctx.malloc(m * 8), ctx.malloc((n * n + n) * 8)
    try:
        ctx.residual_eval(f, pr["x0"], F=Fd, n=n)
        s1, xt1, ss1, _ = ctx.lm_step(f, pr["x0"], None, n, Jd, Fd, Ft, 1e-3, JTJd, jac_mode=AN)
        a = ctx.to_host(JTJd, n * n + n)
        monkeypatch.setenv("PNOL_FUSED_MB", "0.5")               # 2048 rows per block: 15 blocks
        s2, xt2, ss2, _ = ctx.lm_step(f, pr["x0"], None, n, None, Fd, Ft, 1e-3, JTJd, jac_mode=AN)
        b = ctx.to_host(JTJd, n * n + n)
    finally:
        for p in (Jd, Fd, Ft, JTJd):
            ctx.free(p)
    rel = lambda u, v: np.linalg.norm(u - v) / np.linalg.norm(v)   # noqa: E731
    assert rel(b[:n * n], a[:n * n]) < 1e-12 and np.max(np.abs(b[n * n:] - a[n * n:])) < 1e-12 * np.max(np.abs(a[n * n:]))
    assert rel(s2, s1) < 1e-9 and rel(xt2, xt1) < 1e-12 and abs(ss2 - ss1) <= 1e-9 * ss1


# ---------------------------------------------------------------------------------------------------------------------------------
# LM with analytic derivatives
# ---------------------------------------------------------------------------------------------------------------------------------
class Buffers:
    def __init__(self, ctx, m, n):
        self.ctx = ctx
        self.J, self.F, self.Ft, self.JTJ = ctx.malloc(m * n * 8), ctx.malloc(m * 8), ctx.malloc(m * 8), ctx.malloc((n * n + n) * 8)

    def free(self):
        for p in (self.J, self.F, self.Ft, self.JTJ):
            self.ctx.free(p)


def host_rule_step(ctx, f, x, n, m, B, lam, chisq, factor=10.0):
    """pnol_lm_step + the accept / reject rule of Source/LevenbergMarquardtMPI.cpp:107-141 in Python; B.F holds the residuals at x.
    Returns (x, lam, chisq, accepted)"""
    _, xt, ss, _ = ctx.lm_step(f, x, None, n, B.J, B.F, B.Ft, lam, B.JTJ, jac_mode=AN)
    root = math.sqrt(ss)
    chi = root * root
    if chi >= chisq or chi != chi:
        return x, lam * factor, chisq, 0
    ctx.memcpy(B.F, B.Ft, m * 8)
    return xt, lam / factor, chi, 1


def chisq_at(ctx, f, x, n, B):
    """pow(sqrt(sum F^2), 2) at x; leaves F(x) in B.F"""
    _, ss = ctx.residual_eval(f, x, F=B.F, n=n)
    return math.sqrt(ss) * math.sqrt(ss)


def test_lm_iterate_equals_lm_step_and_the_host_rule(ctx, user):
    m, K = 100_000, 8
    pr = problems.lorentz_problem(m, K)
    n = pr["n"]
    f = lorentz(ctx, pr)
    B = Buffers(ctx, m, n)
    try:
        x1, lam1, chi1, seq = pr["x0"].copy(), 1e-3, chisq_at(ctx, f, pr["x0"], n, B), []
        for _ in range(8):
            x1, lam1, chi1, acc = host_rule_step(ctx, f, x1, n, m, B, lam1, chi1)
            seq.append(acc)
        chi0 = chisq_at(ctx, f, pr["x0"], n, B)
        x2, lam2, chi2, acc, rej, _ = ctx.lm_iterate(f, pr["x0"], None, n, B.J, B.F, B.Ft, B.JTJ, 1e-3, chi0, 10.0, 8, jac_mode=AN)
    finally:
        B.free()
    assert np.array_equal(x1, x2) and lam1 == lam2 and chi1 == chi2 and (acc, rej) == (sum(seq), len(seq) - sum(seq))


def np_lm(pr, x0, lam, factor, iters):
    """numpy / scipy restatement of Source/LevenbergMarquardtMPI.cpp:50-141 with the analytic J"""
    t, y, w = pr["t"], pr["y"], pr["w"]

    def resid(x):
        a, c = x[0::2], x[1::2]
        return y - np.sum(a[None, :] / (1.0 + w * (t[:, None] - c[None, :]) ** 2), axis=1)
    x = x0.copy()
    F = resid(x)
    chisq = np.linalg.norm(F) ** 2
    xs, seq, chis = [], [], []
    for _ in range(iters):
        chis.append(chisq)
        J = np_lorentz_grad(x[0::2], x[1::2], w, t)
        JTJ = J.T @ J
        A = JTJ + lam * np.diag(np.diag(JTJ))
        sigma = scipy.linalg.solve(A, -J.T @ F, assume_a="pos")
        Ft = resid(x + sigma)
        chi = np.linalg.norm(Ft) ** 2
        if chi >= chisq or chi != chi:
            lam *= factor
            seq.append(0)
        else:
            lam, chisq, x, F = lam / factor, chi, x + sigma, Ft
            seq.append(1)
        xs.append(x.copy())
    return xs, seq, chis


@pytest.mark.parametrize("m,K,iters", [(100_000, 8, 10), (20_000, 128, 8)])
def test_lm_on_lorentz_problems_matches_numpy_and_converges(ctx, user, m, K, iters):
    pr = problems.lorentz_problem(m, K)
    n = pr["n"]
    f = lorentz(ctx, pr)
    B = Buffers(ctx, m, n)
    try:
        xs_np, seq_np, chis = np_lm(pr, pr["x0"], 1e-3, 10.0, iters)
        x, lam, chisq = pr["x0"].copy(), 1e-3, chisq_at(ctx, f, pr["x0"], n, B)
        for k in range(iters):
            x, lam, chisq, acc = host_rule_step(ctx, f, x, n, m, B, lam, chisq)
            # the decisions agree while chi^2 is far above its rounding noise (zero-noise data: chi^2 -> 0)
            if chis[k] > 1e-16 * chis[0]:
                assert acc == seq_np[k], k
                assert np.max(np.abs(x - xs_np[k])) <= 1e-9 * np.max(np.abs(xs_np[k])), k
        chi0 = chisq_at(ctx, f, pr["x0"], n, B)
        xc, *_ = ctx.lm_iterate(f, pr["x0"], None, n, B.J, B.F, B.Ft, B.JTJ, 1e-3, chi0, 10.0, 40, jac_mode=AN)
    finally:
        B.free()
    assert np.allclose(xc, pr["x_true"], rtol=1e-9, atol=1e-9)


# ---------------------------------------------------------------------------------------------------------------------------------
# the plugin classes, and the refusals
# ---------------------------------------------------------------------------------------------------------------------------------
def test_plugin_classes_with_the_analytic_mode(ctx, user):
    from parallelnonlinearoptimizationlibrary_b200 import hostapi
    hostapi.attach(ctx)
    pr = problems.lorentz_problem(20_000, 16)
    n = pr["n"]
    hostapi.set_jac_mode(AN)
    try:
        r = hostapi.lm_lorentz(pr["t"], pr["y"], pr["w"], pr["x0"], maxiter=30)
        prob = hostapi.LMProblem(pr["t"], pr["y"], pr["w"])
        r2 = prob.run(pr["x0"], maxiter=30)
        prob.close()
        t = np.linspace(-3.0, 5.0, 400)
        truth = np.array([2.5, 1.2, 0.8])
        y = truth[0] * np.exp(-(t - truth[1]) ** 2 * truth[2]) + 0.3
        xg = truth * np.array([1.2, 0.9, 1.1])
        assert user.my_lm_gauss(C.c_void_p(t.ctypes.data), C.c_void_p(y.ctypes.data), C.c_longlong(t.size), C.c_double(0.3),
                                C.c_void_p(xg.ctypes.data), 50) == 0
    finally:
        hostapi.set_jac_mode(capi.JAC_AUTO)
    assert np.allclose(r["X"], pr["x_true"], rtol=1e-9, atol=1e-9) and np.array_equal(r2["X"], r["X"])
    assert np.allclose(xg, truth, rtol=1e-9)
    # the same run as pnol_lm_iterate with the analytic mode
    f = lorentz(ctx, pr)
    B = Buffers(ctx, pr["m"], n)
    try:
        chi0 = chisq_at(ctx, f, pr["x0"], n, B)
        xi, *_ = ctx.lm_iterate(f, pr["x0"], None, n, B.J, B.F, B.Ft, B.JTJ, 1e-3, chi0, 10.0, 30, jac_mode=AN)
    finally:
        B.free()
    assert np.array_equal(r["X"], xi)


@pytest.mark.parametrize("kind", [UJ.MYJ_F_GAUSS_NOJAC, UJ.MYJ_F_GAUSS_V1])
def test_analytic_mode_is_refused_without_a_derivative(ctx, user, kind):
    t = np.linspace(-3.0, 5.0, 3000)
    y = 2.5 * np.exp(-(t - 1.2) ** 2 * 0.8) + 0.3
    x, dx = np.array([2.2, 1.05, 0.9]), np.full(3, 1e-7)
    m, n = t.size, 3
    f = ctx.functor(kind, (0.3,), (), (t, y), m)
    with pytest.raises(capi.PnolError, match="NO_FUNCTOR.*no analytic Jacobian"):
        ctx.fd_jacobian(f, x, None, mode=AN)
    B = Buffers(ctx, m, n)
    try:
        _, ss = ctx.residual_eval(f, x, F=B.F, n=n)
        for J in (B.J, None):
            with pytest.raises(capi.PnolError, match="NO_FUNCTOR"):
                ctx.lm_step(f, x, None, n, J, B.F, B.Ft, 1e-3, B.JTJ, jac_mode=AN)
            with pytest.raises(capi.PnolError, match="NO_FUNCTOR"):
                ctx.lm_iterate(f, x, None, n, J, B.F, B.Ft, B.JTJ, 1e-3, ss, 10.0, 3, jac_mode=AN)
    finally:
        B.free()
    # AUTO on the same model: the forward difference, bit for bit the host's quotients (Source/PNOL_Objective.cpp:186-192)
    J, F = ctx.fd_jacobian(f, x, dx)
    _, Fh = UJ.host_jacobian(UJ.MYJ_F_GAUSS, (0.3,), (t, y), x)
    assert np.array_equal(F, Fh)
    for j in range(n):
        xj = x.copy()
        xj[j] = xj[j] + dx[j]
        _, Fj = UJ.host_jacobian(UJ.MYJ_F_GAUSS, (0.3,), (t, y), xj)
        assert np.array_equal(J[:, j], (Fj - Fh) / dx[j])
