"""The linear algebra of the Levenberg-Marquardt step against exact and extended-precision references (tests/exact_reference.py):
J^T J / J^T F bit for bit on graded integer inputs, J^T F of the LM step bit for bit through one-hot residuals, the Cholesky solve
over its whole range n = 1 ... 704 against backward- and forward-error bars, its pivot range, and the LM step at n = 128 and 512."""
import ctypes as C

import numpy as np
import pytest

import exact_reference as R
import oracle_lib as O
from parallelnonlinearoptimizationlibrary_b200 import capi, problems
from test_gpu_parity_core import _lm_python_loop, rel

pytestmark = pytest.mark.gpu

U = R.U


# ---- (a) normal equations on graded integer J: exact ------------------------------------------------------------------------------

NORMAL_EQ_SHAPES = [(1, 32), (31, 16), (33, 128), (64, 256), (4737, 256), (100_000, 48), (7000, 272), (5000, 512),
                    (300_000, 256), (2000, 144), (513, 192), (40, 240), (700, 4096), (300, 8192), (4_000_000, 256)]


def _periodic_to_device(ctx, base, m):
    """device copy of the m rows base[i mod P] (base: P x w, C order), by doubling device-to-device copies"""
    P = base.shape[0]
    row = base[0].nbytes
    p = ctx.malloc(m * row)
    ctx.memcpy(p, np.ascontiguousarray(base[:min(P, m)]), min(P, m) * row)
    k = P
    while k < m:                                   # rows [0, k) are in place and k is a multiple of P
        c = min(k, m - k)
        ctx.memcpy(p + k * row, p, c * row)
        k += c
    return p


def _check_normal_eq(JTJ, A, rhs, JTJw, rhsw, lam):
    n = JTJw.shape[0]
    assert np.array_equal(JTJ, JTJw), "J^T J: %d entries differ" % np.count_nonzero(JTJ != JTJw)
    off = ~np.eye(n, dtype=bool)
    assert np.array_equal(A[off], JTJw[off])
    assert np.array_equal(np.diag(A), (1 + lam) * np.diag(JTJw))
    assert np.array_equal(rhs, rhsw), "rhs: %d entries differ" % np.count_nonzero(rhs != rhsw)


@pytest.mark.parametrize("m,n", NORMAL_EQ_SHAPES)
def test_normal_eq_bit_exact_on_graded_integers(ctx, m, n):
    # every tile role, the ragged last chunk (the TMA's zero fill), the mirroring, the stream-K kernel (with F) and the CTA-pair
    # kernel (without F, two tile rows: n = 144 ... 256): all exact, so every summation order gives the same bits
    rng = np.random.default_rng(11 * m + n)
    lam = 0.25
    periodic = m > 1_000_000
    g = R.periodic_graded_matrix(m, n, rng) if periodic else R.graded_integer_matrix(m, n, rng)
    JTJw, rhsw = g.jtj(), -g.jtf()
    if periodic:
        Jd = _periodic_to_device(ctx, g.K.astype(np.float64) * g.scale, m)
        Fd = _periodic_to_device(ctx, g.F.astype(np.float64)[:, None], m)
    else:
        J, F = g.J, g.F.astype(np.float64)
        _check_normal_eq(*ctx.lm_normal_eq(J, F, m, n, lam), JTJw, rhsw, lam)          # host arrays
        Jd, Fd = ctx.to_device(J), ctx.to_device(F)
    outs = [ctx.malloc(n * n * 8), ctx.malloc(n * n * 8), ctx.malloc(n * 8)]
    try:
        for with_f in (True, False):
            ctx.lm_normal_eq(Jd, Fd if with_f else None, m, n, lam, JTJ=outs[0], A=outs[1], rhs=outs[2])
            got = [ctx.to_host(outs[0], (n, n)), ctx.to_host(outs[1], (n, n)), ctx.to_host(outs[2], n)]
            _check_normal_eq(*got, JTJw, rhsw if with_f else np.zeros(n), lam)
    finally:
        for p in [Jd, Fd] + outs:
            ctx.free(p)


# ---- (b) J^T F of the LM step through one-hot residuals ---------------------------------------------------------------------------

K_ONEHOT = 128
ROUND_WARPS_PER_SM = 16          # the structured Jacobian kernel's grid on the B200: 2 blocks of 8 warps per SM (DESIGN.md section 4)


def _special_problem(m, K):
    """the Lorentz problem with two rows outside the branch-free range: t = 1e200 (its J row is zero) and y = 1e-70 (below 2^-200:
    the row takes the `/` path with a nonzero J row). Returns (pr, special rows)."""
    pr = problems.lorentz_problem(m, K)
    s = [m // 3, m // 3 + 1]
    pr["t"] = pr["t"].copy()
    pr["y"] = pr["y"].copy()
    pr["t"][s[0]] = 1e200
    pr["y"][s[1]] = 1e-70
    return pr, s


def _onehot_rows(m, nwarps, special, rng, nrandom):
    rows = {0, 31, 32, m - 1} | set(special)
    nbatch = (m + 31) // 32
    full = nbatch // nwarps
    if full >= 1:
        rows.add(nwarps * 32 if full >= 2 else 0)              # first row of round 2
        covered = full * nwarps * 32                            # start of the ragged remainder
        rows.update(range(max(covered - 3, 0), min(covered + 4, m)))
    rows.update(rng.integers(0, m, size=nrandom).tolist())
    return sorted(r for r in rows if 0 <= r < m)


def _set_f(ctx, Fd, m, entries):
    ctx.check(ctx.lib.pnol_memset(ctx.h, C.c_void_p(Fd), 0, C.c_size_t(m * 8)))
    for i, v in entries:
        ctx.memcpy(Fd + 8 * i, np.array([v]), 8)


ONEHOT_CASES = [(m, mode) for m in (2000 + K_ONEHOT, 2 * 75_776, 500_000, 4_000_000) for mode in ("structured",)] + \
               [(m, mode) for m in (2000 + K_ONEHOT, 500_000) for mode in ("blackbox", "rowblocked")]


@pytest.mark.parametrize("dx0", [1e-7, 1e-5])
@pytest.mark.parametrize("m,mode", ONEHOT_CASES)
def test_lm_step_jtf_bit_exact_through_one_hot_residuals(ctx, m, mode, dx0, monkeypatch):
    # The Jacobian kernels compute their own residuals at x; the F handed to pnol_lm_step only enters J^T F. With F = e_i every term
    # of J^T F but one is an exact zero, so -J^T F = -J[i, :] bit for bit whatever the order, on every path: the 32-row batches dealt
    # round-robin, the ragged remainder split evenly, the `/` fallback rows, the black-box SYRK F tiles, the row blocks.
    # dX = 1e-7 takes the three-operation FD quotient, 1e-5 the five-operation one (exact_div.cuh).
    K = K_ONEHOT
    pr, special = _special_problem(m, K)
    n = pr["n"]
    f = ctx.functor(capi.F_LORENTZ_SUM, (pr["w"],), (), (pr["t"], pr["y"]), m)
    dx = np.full(n, dx0)
    rng = np.random.default_rng(m + int(dx0 * 1e7))
    nwarps = ROUND_WARPS_PER_SM * ctx.sm_count
    rows = _onehot_rows(m, nwarps, special, rng, 30 if mode == "structured" else 6)
    Jd = ctx.malloc(m * n * 8)
    Fd, Ft, JTJd = ctx.malloc(m * 8), ctx.malloc(m * 8), ctx.malloc((n * n + n) * 8)
    try:
        if mode == "rowblocked":
            monkeypatch.setenv("PNOL_FUSED_MB", str(max(1, m * n * 8 // (5 << 20))))       # five row blocks or so
            ctx.fd_jacobian(f, pr["x0"], dx, J=Jd, F=Ft)                                  # the reference rows of J
        jac_mode = capi.JAC_BLACKBOX if mode == "blackbox" else capi.JAC_AUTO
        Jarg = None if mode == "rowblocked" else Jd

        def rhs_for(entries):
            _set_f(ctx, Fd, m, entries)
            _, _, _, info = ctx.lm_step(f, pr["x0"], dx, n, Jarg, Fd, Ft, 1e-3, JTJd, jac_mode=jac_mode)
            return ctx.to_host(JTJd + n * n * 8, n)

        def jrow(i):
            return ctx.to_host(Jd + i * n * 8, n)

        for i in rows:
            got = rhs_for([(i, 1.0)])
            assert np.array_equal(got, -jrow(i)), "row %d: %d entries differ" % (i, np.count_nonzero(got != -jrow(i)))
        assert np.any(jrow(special[1])) and not np.any(jrow(special[0]))       # the fallback rows are what they claim
        pairs = [(0, m - 1), (31, 32), (special[0], special[1])] + [tuple(rng.integers(0, m, size=2)) for _ in range(3)]
        for i, j in pairs:
            if i == j:
                continue
            got = rhs_for([(i, 1.0), (j, 1.0)])
            assert np.array_equal(got, -(jrow(i) + jrow(j))), (i, j)
    finally:
        for p in (Jd, Fd, Ft, JTJd):
            ctx.free(p)
        f.close()


# ---- (c) the solve over its whole range --------------------------------------------------------------------------------------------

def _solve_raw(ctx, A, b, n):
    """pnol_spd_solve without raising: (status, info, x, message)"""
    A, b = np.ascontiguousarray(A, dtype=np.float64), np.ascontiguousarray(b, dtype=np.float64)
    x = np.zeros(n)
    info = C.c_int(-1)
    st = ctx.lib.pnol_spd_solve(ctx.h, capi._ptr(A), capi._ptr(b), int(n), capi._ptr(x), C.byref(info))
    msg = ctx.lib.pnol_last_error(ctx.h)
    return st, info.value, x, (msg.decode() if msg else "")


def _bars(A, x, b, D, kappa, n, xref=None):
    """(eta, forward error, forward bar)"""
    xref = R.refined_solution(A, b) if xref is None else xref
    return R.backward_error(A, x, b), R.forward_error(x, xref, D), 4 * n * U * kappa


def _lm_family(ctx, n):
    K, m = n // 2, max(3 * n, 64)
    pr = problems.lorentz_problem(m, K)
    f = ctx.functor(capi.F_LORENTZ_SUM, (pr["w"],), (), (pr["t"], pr["y"]), m)
    J, _ = ctx.fd_jacobian(f, pr["x0"], np.full(n, 1e-7))
    f.close()
    return J.T @ J


@pytest.mark.parametrize("family", R.FAMILIES + ("lm",))
def test_spd_solve_meets_the_error_bars_over_its_whole_range(ctx, family):
    # eta <= n u and ||x - x_ref|| <= 4 n u kappa_2(A) ||x_ref|| (graded D C D: in the D-scaled norm, with kappa_2(C)), x_ref the
    # Cholesky solution refined with long-double residuals. n: every n in 1..80, n = -1..3 mod 32 up to 704, both buffer plans of
    # the back substitution (n <= 416: double-buffered; from 417 on: one buffer)
    rng = np.random.default_rng(12)
    misses = []
    cases = []
    if family == "lm":
        for n in R.LM_SIZES:
            JTJ = _lm_family(ctx, n)
            b = rng.normal(size=n)
            for lam in R.LM_LAMBDAS:
                A = R.lm_like(JTJ, lam)
                cases.append((n, A, b, None, R.kappa2(A), lam))
    else:
        cases = ((n,) + R.spd_family(family, n, rng) + (None,) for n in R.solve_sizes())
    for n, A, b, D, kappa, tag in cases:
        x = ctx.spd_solve(A, b, n)
        eta, fwd, fbar = _bars(A, x, b, D, kappa, n)
        if not (eta <= n * U and fwd <= fbar):
            import scipy.linalg
            xs = scipy.linalg.cho_solve(scipy.linalg.cho_factor(A, lower=True), b)
            misses.append("n=%d %s: eta %.3g (n u %.3g, scipy %.3g), forward %.3g (bar %.3g)"
                          % (n, tag, eta, n * U, R.backward_error(A, xs, b), fwd, fbar))
    assert not misses, "\n".join(misses)


@pytest.mark.parametrize("n", [1, 2, 3, 31, 32, 33, 100, 416, 417, 511, 512, 513, 703, 704])
def test_spd_solve_exact_properties(ctx, n):
    rng = np.random.default_rng(13 + n)
    A, b, _, _ = R.spd_family("random", n, rng, want_kappa=False)
    x = ctx.spd_solve(A, b, n)
    assert np.array_equal(ctx.spd_solve(A, b, n), x)                                 # deterministic
    Au = A.copy()
    Au[np.triu_indices(n, 1)] = np.nan                                              # only the lower triangle is read
    assert np.array_equal(ctx.spd_solve(Au, b, n), x)
    if n % 4 == 0:
        # A at a device address 8 bytes past 32-byte alignment: the scalar-load path, same bits as the 256-bit path
        base, bd, xd = ctx.malloc((n * n + 4) * 8), ctx.to_device(b), ctx.malloc(n * 8)
        try:
            Ad = ctx.to_device(A)
            ctx.memcpy(base + 8, A, A.nbytes)
            ctx.spd_solve(Ad, bd, n, x=xd)
            xa = ctx.to_host(xd, n)
            ctx.spd_solve(base + 8, bd, n, x=xd)
            assert np.array_equal(ctx.to_host(xd, n), xa)
            ctx.free(Ad)
        finally:
            for p in (base, bd, xd):
                ctx.free(p)
    # A scaled by 4^200 and 4^-200: the same bars; every operation scales exactly (powers of 4 keep the square roots exact)
    for e in (200, -200):
        s = 4.0 ** e
        xs = ctx.spd_solve(A * s, b, n)
        eta, fwd, fbar = _bars(A * s, xs, b, None, R.kappa2(A), n)
        assert eta <= n * U and fwd <= fbar, (e, eta, fwd, fbar)
        assert np.array_equal(xs * s, x), "4^%d: not bit-identical to the unscaled solve" % e


def test_spd_solve_rejects_n_outside_its_range(ctx):
    with pytest.raises(capi.PnolError, match="INVALID"):
        ctx.spd_solve(np.eye(705), np.ones(705), 705)
    st, _, _, _ = _solve_raw(ctx, np.eye(705), np.ones(705), 705)
    assert st == capi.ERR_INVALID


@pytest.mark.parametrize("k", [1, 31, 32, 33, 416, 417, 700])
def test_spd_solve_not_spd_names_the_pivot(ctx, k):
    n = 704
    A = R.ldl_indefinite(n, k, np.random.default_rng(k))
    st, info, x, msg = _solve_raw(ctx, A, np.ones(n), n)
    assert st == 5 and info == k + 1 and ("pivot %d " % (k + 1)) in msg, (st, info, msg)
    assert np.all(np.isnan(x))


@pytest.mark.parametrize("n,k", [(1, 0), (40, 39), (40, 5), (417, 416), (417, 100)])
def test_spd_solve_rejects_a_subnormal_pivot(ctx, n, k):
    # a subnormal pivot passes `d > 0`, and rcp.approx.ftz / rsqrt.approx.ftz flush it to zero: it must be rejected at its own
    # column (not one later after a NaN, and not accepted with a NaN solution when it is the last pivot)
    for d in (2.0 ** -1040, 2.0 ** -1074, np.nextafter(2.0 ** -1022, 0)):
        A = np.eye(n)
        A[k, k] = d
        st, info, x, msg = _solve_raw(ctx, A, np.ones(n), n)
        assert (st, info) == (5, k + 1), "d = %r: status %d, info %d (%s)" % (d, st, info, msg)
        assert np.all(np.isnan(x))


@pytest.mark.parametrize("n,k", [(1, 0), (40, 39), (40, 5), (417, 300)])
def test_spd_solve_pivot_range_edges(ctx, n, k):
    for d in (2.0 ** 1000, np.inf, np.nan, 0.0, -0.0):
        A = np.eye(n)
        A[k, k] = d
        st, info, x, _ = _solve_raw(ctx, A, np.ones(n), n)
        assert (st, info) == (5, k + 1), d
    # the smallest normal and the largest accepted pivot solve
    for d in (2.0 ** -1022, np.nextafter(2.0 ** 1000, 0)):
        A = np.eye(n)
        A[k, k] = d
        st, info, x, _ = _solve_raw(ctx, A, np.ones(n), n)
        want = np.ones(n)
        want[k] = 1 / d
        assert (st, info) == (0, 0) and np.all(np.isfinite(x)) and np.max(np.abs(x - want) / want) <= 8 * U, d


# ---- (d) the LM step at n = 128 and n = 512 ----------------------------------------------------------------------------------------

@pytest.mark.parametrize("K", [64, 256])
def test_lm_step_solve_and_trial_point_at_n_128_and_512(ctx, K):
    m = 2000 + K
    pr = problems.lorentz_problem(m, K)
    t = pr["t"].copy()
    t[[7, m // 2]] = (1e200, 1e30)           # residual rows outside the branch-free range (the second with nonzero terms)
    n = pr["n"]
    f = ctx.functor(capi.F_LORENTZ_SUM, (pr["w"],), (), (t, pr["y"]), m)
    of = O.OFunctor(capi.F_LORENTZ_SUM, (pr["w"],), (), (t, pr["y"]), m)
    dx = np.full(n, 1e-7)
    lam = 1e-3
    x0 = pr["x0"]
    F0, _ = ctx.residual_eval(f, x0)
    assert np.array_equal(F0, O.residual(of, x0))                        # lorentz_rowwise_kernel<64> / <256>
    Jd, Fd, Ft, JTJd = ctx.malloc(m * n * 8), ctx.malloc(m * 8), ctx.malloc(m * 8), ctx.malloc((n * n + n) * 8)
    try:
        ctx.residual_eval(f, x0, F=Fd, n=n)
        sigma, xt, ss, info = ctx.lm_step(f, x0, dx, n, Jd, Fd, Ft, lam, JTJd)
        assert info == 0
        packed = ctx.to_host(JTJd, n * n + n)
        A, rhs = R.lm_like(packed[:n * n].reshape(n, n), lam), packed[n * n:]
        assert np.array_equal(sigma, ctx.spd_solve(A, rhs, n))
        eta, fwd, fbar = _bars(A, sigma, rhs, None, R.kappa2(A), n)
        assert eta <= n * U and fwd <= fbar, (eta, fwd, fbar)
        assert np.array_equal(xt, x0 + sigma)
        Fw = O.residual(of, xt)
        assert np.array_equal(ctx.to_host(Ft, m), Fw)
        Fr, ssr = ctx.residual_eval(f, xt)
        assert np.array_equal(Fr, Fw) and ss == ssr
    finally:
        for p in (Jd, Fd, Ft, JTJd):
            ctx.free(p)


@pytest.mark.parametrize("K", [64, 256])
def test_lm_iterates_match_oracle_at_n_128_and_512(ctx, K):
    m, iters = 2000 + K, 5
    pr = problems.lorentz_problem(m, K)
    f = ctx.functor(capi.F_LORENTZ_SUM, (pr["w"],), (), (pr["t"], pr["y"]), m)
    of = O.OFunctor(capi.F_LORENTZ_SUM, (pr["w"],), (), (pr["t"], pr["y"]), m)
    want = O.lm(of, pr["x0"], 0.001, 10.0, 1e-7, iters, 0.0, want_trace=True)
    X, trace, it = _lm_python_loop(ctx, f, pr["x0"], m, 0.001, 10.0, 1e-7, iters, 0.0)
    assert it == want["iters"]
    wt = want["trace"][:trace.shape[0]]
    n = pr["n"]
    assert np.array_equal(trace[:, n + 1], wt[:, n + 1])                 # accept / reject history identical
    for k in range(trace.shape[0]):
        assert rel(trace[k, :n], wt[k, :n]) < 1e-9, "iterate %d: %.3g" % (k, rel(trace[k, :n], wt[k, :n]))
    assert rel(X, want["X"]) < 1e-9
    assert abs(trace[-1, n] - want["chisq"]) <= 1e-9 * max(want["chisq"], 1e-30) + 1e-24
