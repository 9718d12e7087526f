"""The checkers of tests/test_gpu_lm_linear_algebra.py and tests/test_gpu_dense_exact.py, checked on the CPU: the integer
constructions make numpy's float64 J^T J / J^T F, p = -D g, A B and both forms of updateHessianInv exact (equal to integer arithmetic
bit for bit), an exact comparison notices what the old norm-wise bars do not, the solve's bars (backward error eta <= n u,
tests/exact_reference.py) are met by scipy's own solution and missed by small perturbations, the componentwise bars of the dense
kernels are missed when one term of one sum is dropped, and the GPU cases reach every branch of the launchers."""
import numpy as np
import pytest
import scipy.linalg

import exact_reference as R
import oracle_lib as O
from parallelnonlinearoptimizationlibrary_b200 import capi, problems

# the shapes of test_lm_normal_eq_stream_k_shapes (tests/test_gpu_parity_core.py), i.e. the largest row count the GPU tests use
# at every n
NORMAL_EQ_SHAPES = [(1, 32), (31, 16), (33, 128), (64, 256), (4737, 256), (100_000, 48), (7000, 272), (5000, 512),
                     (300_000, 256), (2000, 144), (513, 192), (40, 240), (700, 4096), (300, 8192)]
FULL_INT_WORK = 2e7                  # m n^2 up to which the whole K^T K is also formed in int64 (numpy's int matmul is not BLAS)


def _pairs(n, rng, count=300):
    """diagonal, tile corners and random (j, l) pairs of the lower triangle"""
    idx = {(j, j) for j in range(n)}
    for c in (0, 127, 128, 255, 256, n - 1):
        if c < n:
            idx.update({(c, 0), (n - 1, c), (c, c // 2)})
    j = rng.integers(0, n, size=count)
    l = rng.integers(0, n, size=count)
    idx.update(zip(np.maximum(j, l).tolist(), np.minimum(j, l).tolist()))
    return sorted(idx)


def _check_exact(g, rng, m, n):
    JTJ = g.jtj()
    assert np.array_equal(JTJ, JTJ.T)
    if m * n * n <= FULL_INT_WORK:
        G = g.K.T @ (g.K * g.counts[:, None]) if g.counts is not None else g.K.T @ g.K
        assert np.array_equal(JTJ, G.astype(np.float64) * np.outer(g.scale, g.scale))
    for j, l in _pairs(n, rng):
        v = g.jtj_int_entry(j, l)
        assert abs(v) < 2 ** 53
        assert JTJ[j, l] == np.ldexp(float(v), -int(g.s[j] + g.s[l])), (j, l)
    jtf_int = g.jtf_int()
    assert np.all(np.abs(jtf_int) < 2 ** 53)
    assert np.array_equal(g.jtf(), jtf_int.astype(np.float64) * g.scale)
    return JTJ


@pytest.mark.parametrize("m,n", NORMAL_EQ_SHAPES)
def test_blas_product_of_graded_integer_matrix_is_exact(m, n):
    rng = np.random.default_rng(1000 + n)
    g = R.graded_integer_matrix(m, n, rng)
    assert m * 4 ** R.integer_bits(m) < 2 ** 53
    assert set(g.s[:128].tolist()) != {g.s[0]}                        # the first tile mixes scales
    _check_exact(g, rng, m, n)
    # the same numbers through the materialised J (what the GPU test hands the kernel)
    J = g.J
    if m * n * n <= 1e10:
        assert np.array_equal(J.T @ J, g.jtj())
        assert np.array_equal(J.T @ g.F.astype(np.float64), g.jtf())


def test_periodic_4m_construction_is_exact():
    m, n = 4_000_000, 256
    rng = np.random.default_rng(4)
    g = R.periodic_graded_matrix(m, n, rng)
    assert g.counts.sum() == m and m * 4 ** R.integer_bits(m) < 2 ** 53
    _check_exact(g, rng, R.PERIOD, n)
    # materialised at a width the host can afford: the count-weighted product equals the plain product of all 4M rows
    g8 = R.periodic_graded_matrix(m, 8, np.random.default_rng(5))
    J, F = R.periodic_rows(g8, 0, m)
    assert np.array_equal(J.T @ J, g8.jtj()) and np.array_equal(J.T @ F, g8.jtf())
    # and a window that starts inside the period
    Jw, Fw = R.periodic_rows(g8, 4098, 4098 + 3)
    assert np.array_equal(Jw[1], g8.K[0] * g8.scale) and Fw[1] == g8.F[0]


def test_exact_comparison_notices_what_the_norm_bar_does_not():
    m, n = 4737, 256
    rng = np.random.default_rng(6)
    g = R.graded_integer_matrix(m, n, rng)
    J, JTJ = g.J, g.jtj()
    # a dropped row (a chunk boundary that loses a row): any row with a nonzero entry changes J^T J exactly
    i = int(np.flatnonzero(np.any(g.K != 0, axis=1))[m // 2])
    Jd = np.delete(J, i, axis=0)
    assert not np.array_equal(Jd.T @ Jd, JTJ)
    assert not np.array_equal(Jd.T @ np.delete(g.F, i).astype(np.float64), g.jtf())
    # one entry off by one ulp -- in the smallest-scale column, where 1e-12 norm-wise cannot see it
    small = int(np.flatnonzero((g.s == R.SCALE_MAX) & np.any(g.K != 0, axis=0))[0])
    bad = JTJ.copy()
    bad[small, small] = np.nextafter(bad[small, small], np.inf)
    assert not np.array_equal(bad, JTJ)
    assert np.linalg.norm(bad - JTJ) <= 1e-12 * np.linalg.norm(JTJ)
    # so is a whole small-scale column that is wrong by far more than an ulp
    bad[:, small] *= 1 + 1e-6
    assert np.linalg.norm(bad - JTJ) <= 1e-12 * np.linalg.norm(JTJ)


def _lm_jtj(n):
    """J^T J of the Lorentz problem at K = n / 2 (the oracle's Jacobian: bit-identical to the device's, test_gpu_parity_core.py)"""
    K = n // 2
    m = max(3 * n, 64)
    pr = problems.lorentz_problem(m, K)
    of = O.OFunctor(capi.F_LORENTZ_SUM, (pr["w"],), (), (pr["t"], pr["y"]), m)
    J, _ = O.fd_jacobian(of, pr["x0"], np.full(n, 1e-7))
    return J.T @ J


@pytest.mark.parametrize("family", R.FAMILIES)
def test_scipy_solution_meets_the_backward_error_bar(family):
    rng = np.random.default_rng(7)
    for n in R.solve_sizes():
        A, b, _, _ = R.spd_family(family, n, rng, want_kappa=False)
        x = scipy.linalg.cho_solve(scipy.linalg.cho_factor(A, lower=True), b)
        eta = R.backward_error(A, x, b)
        assert eta <= n * R.U, (n, eta)


def test_scipy_solution_meets_the_backward_error_bar_lm_like():
    rng = np.random.default_rng(8)
    for n in R.LM_SIZES:
        JTJ = _lm_jtj(n)
        b = rng.normal(size=n)
        for lam in R.LM_LAMBDAS:
            A = R.lm_like(JTJ, lam)
            x = scipy.linalg.cho_solve(scipy.linalg.cho_factor(A, lower=True), b)
            eta = R.backward_error(A, x, b)
            assert eta <= n * R.U, (n, lam, eta)


def test_perturbed_solutions_miss_the_bar():
    # b = A x_true, so that ||A x|| is comparable with ||A|| ||x||: a relative change of x shows in the residual
    rng = np.random.default_rng(9)
    for n in R.solve_sizes():
        A, _, _, _ = R.spd_family("random", n, rng, want_kappa=False)
        b = A @ rng.uniform(1, 2, size=n)
        x = R.refined_solution(A, b)
        assert R.backward_error(A, x, b) <= n * R.U
        assert R.backward_error(A, x * (1 + 1e-11), b) > n * R.U, n
        j = int(np.argmax(np.abs(x)))
        y = x.copy()
        y[j] *= 1 + 1e-10
        assert R.backward_error(A, y, b) > n * R.U, n


def test_refined_solution_has_the_smallest_residual():
    # Q diag(geomspace(1, 1e-12)) Q^T: refinement with long-double residuals leaves a backward error at the float64 rounding of x
    rng = np.random.default_rng(10)
    n = 200
    A, b, _, _ = R.spd_family("geometric", n, rng, want_kappa=False)
    x = R.refined_solution(A, b)
    xl = scipy.linalg.cho_solve(scipy.linalg.cho_factor(A, lower=True), b)
    assert R.backward_error(A, x, b) <= min(R.backward_error(A, xl, b), 2 * R.U)


def test_solve_sizes_cover_both_buffer_plans_and_every_ragged_block():
    s = R.solve_sizes()
    assert s[:80] == list(range(1, 81)) and s[-1] == 704 and 705 not in s
    assert {416, 417, 511, 512, 513, 703, 704} <= set(s)
    assert {v % 32 for v in s} == set(range(32)) and any(v % 4 for v in s if v > 416)


# ---- the dense BFGS pieces and the DMMA GEMM (tests/test_gpu_dense_exact.py) ---------------------------------------------------

import test_gpu_dense_exact as T      # noqa: E402  (its case tables and path restatement; the module's tests need a GPU)


def _rel(a, b):
    return np.linalg.norm(a - b) / np.linalg.norm(b)


def _one_ulp_off(want):
    """want with its smallest nonzero entry moved by one ulp"""
    bad = want.copy()
    flat = bad.reshape(-1)
    nz = np.flatnonzero(flat)
    i = nz[np.argmin(np.abs(flat[nz]))]
    flat[i] = np.nextafter(flat[i], np.inf)
    return bad


@pytest.mark.parametrize("n", [1, 5, 128, 516, 4096, 4100])
def test_graded_matvec_is_exact(n):
    c = R.GradedMatvec(n, np.random.default_rng(n))
    assert c.peak < 2 ** 53
    assert np.array_equal(-(c.D @ c.g), c.want)                          # BLAS order: exact by the bound
    assert np.array_equal(-(c.D[:, ::-1] @ c.g[::-1]), c.want)           # and in the reverse order
    assert np.array_equal(np.ldexp(c.want, c.r), -(c.K @ c.G).astype(np.float64))
    if n >= 128:
        # exponents mix inside every 4-wide lane group and every 128-column group; zero rows and columns are present
        groups = c.t[:n - n % 4].reshape(-1, 4)
        assert all(len(set(q)) > 1 for q in groups.tolist())
        assert len(set(c.t[:128].tolist())) > 30
        assert np.any(~c.K.any(axis=1)) and np.any(~c.K.any(axis=0))
    bad = _one_ulp_off(c.want)
    assert not np.array_equal(bad, c.want) and _rel(bad, c.want) < 1e-13


@pytest.mark.parametrize("M,N,K", [(1, 1, 1), (129, 257, 512), (300, 130, 65), (127, 2, 33)])
def test_graded_gemm_is_exact(M, N, K):
    c = R.GradedGemm(M, N, K, np.random.default_rng(M + N + K))
    assert c.peak < 2 ** 53
    KL = c.Ka @ c.Lb                                                     # int64, not BLAS
    assert np.array_equal(c.int_product_f64(), KL.astype(np.float64))
    assert np.array_equal(c.A @ c.B, c.want()) and np.array_equal(c.want(), c.want(KL.astype(np.float64)))
    bad = _one_ulp_off(c.want())
    assert not np.array_equal(bad, c.want()) and _rel(bad, c.want()) < 1e-13


def test_every_gpu_construction_stays_below_2_53():
    for n, *_ in T.MATVEC_CASES:
        assert R.GradedMatvec(n, np.random.default_rng(n)).peak < 2 ** 53
    for M, N, K, *_ in T.GEMM_CASES + [T.GEMM_BIG + (0, 0, 0)]:
        assert R.GradedGemm(M, N, K, np.random.default_rng(1)).peak < 2 ** 53
    for n, k, sign, oD, og, os_ in T.HINV_CASES:
        c = R.IntegerHinv(n, k, sign, np.random.default_rng(200 + n + oD + 2 * og + 3 * os_))     # the GPU test's seed
        assert c.peak < 2 ** 53, (n, k, sign)


def _numpy_hinv_forms(c):
    rho = c.sign * 2.0 ** -c.k
    D, g, s = c.D, c.g, c.s
    M1, M2 = np.eye(c.n) - rho * np.outer(s, g), np.eye(c.n) - rho * np.outer(g, s)
    literal = (M1 @ D) @ M2 + rho * np.outer(s, s)
    u, v = D @ g, D.T @ g
    rank2 = D + (-rho * np.outer(s, v) - rho * np.outer(u, s) + (rho * rho * (g @ u) + rho) * np.outer(s, s))
    return literal, rank2


@pytest.mark.parametrize("n,k,sign", [(1, 0, 1), (6, 0, 1), (6, 3, -1), (257, 2, 1), (1024, 3, -1), (4096, 1, 1)])
def test_integer_hinv_is_exact_in_both_forms(n, k, sign):
    c = R.IntegerHinv(n, k, sign, np.random.default_rng(n + k))
    assert c.peak < 2 ** 53 and int(c.gi @ c.si) == sign * 2 ** k
    literal, rank2 = _numpy_hinv_forms(c)
    assert np.array_equal(rank2, c.want)
    if n <= 1024:                                                         # two n^3 products on the host
        assert np.array_equal(literal, c.want)
    bad = _one_ulp_off(c.want)
    assert not np.array_equal(bad, c.want) and _rel(bad, c.want) < 1e-12


def test_uv_swap_is_seen_only_with_a_nonsymmetric_d():
    rng = np.random.default_rng(14)
    sym = R.IntegerHinv(64, 2, 1, rng, symmetric=True)
    assert np.array_equal(sym.Di, sym.Di.T) and np.array_equal(sym.swapped(), sym.want)
    for n in (6, 257):
        c = R.IntegerHinv(n, 2, -1, rng)
        assert not np.array_equal(c.swapped(), c.want)


# ---- the componentwise bars: met by the rounded reference, missed with one term of one sum dropped -------------------------------

def _median_term(x):
    """index of the median-magnitude nonzero entry"""
    nz = np.flatnonzero(x)
    return nz[np.argsort(np.abs(x[nz]))[nz.size // 2]]


@pytest.mark.parametrize("graded", [False, True])
@pytest.mark.parametrize("n,path", [(129, "scalar"), (4096, "v4"), (4098, "scalar")])
def test_matvec_bar_misses_a_dropped_term(n, path, graded):
    rng = np.random.default_rng(400 + n)
    D, g = rng.normal(size=(n, n)), rng.normal(size=n)
    if graded:
        D = D * np.outer(R.graded_scaling(n), R.graded_scaling(n))
    assert R.matvec_path(n) == path
    ref, bar = R.matvec_bar(D, g, R.matvec_depth(n, path))
    assert R.within(ref.astype(np.float64), ref, bar)
    i = n // 2
    k = _median_term(D[i] * g)
    bad = ref.copy()
    bad[i] += R.ld(D[i, k]) * R.ld(g[k])                                  # p_i = -sum: the term left out
    assert not R.within(bad.astype(np.float64), ref, bar)


@pytest.mark.parametrize("graded", [False, True])
@pytest.mark.parametrize("M,N,K", [(129, 127, 65), (128, 130, 4096)])
def test_gemm_bar_misses_a_dropped_term(M, N, K, graded):
    rng = np.random.default_rng(500 + M + N + K)
    A, B = rng.normal(size=(M, K)), rng.normal(size=(K, N))
    if graded:
        A, B = A * R.graded_scaling(M)[:, None], B * R.graded_scaling(N)[None, :]
    ref, bar = R.gemm_bar(A, B, R.gemm_depth(K))
    assert R.within(ref.astype(np.float64), ref, bar)
    i, j = M // 2, N // 2
    k = _median_term(A[i] * B[:, j])
    bad = ref.copy()
    bad[i, j] -= R.ld(A[i, k]) * R.ld(B[k, j])
    assert not R.within(bad.astype(np.float64), ref, bar)


@pytest.mark.parametrize("graded", [False, True])
@pytest.mark.parametrize("n", [130, 1024])
def test_hinv_bar_misses_a_dropped_term(n, graded):
    rng = np.random.default_rng(600 + n)
    D, g = rng.normal(size=(n, n)), rng.normal(size=n)
    if graded:
        D = D * np.outer(R.graded_scaling(n), R.graded_scaling(n))
    s = 0.1 * g + 0.05 * rng.normal(size=n)
    path = R.hinv_rank2_path(n)
    ref, Tm, kappa = R.hinv_reference_ld(D, g, s)
    bar = R.hinv_bar(n, Tm, kappa, *R.hinv_depths(n, path, 148))
    assert R.within(ref.astype(np.float64), ref, bar)
    i = n // 2
    k = _median_term(D[i] * g)
    for which in ("u", "v"):
        # the update with one term missing from u_i = sum_k D_ik g_k (or from v_i = sum_k D_ki g_k)
        Dl, gl, sl = R.ld(D), R.ld(g), R.ld(s)
        u, v = Dl @ gl, Dl.T @ gl
        if which == "u":
            u[i] -= Dl[i, k] * gl[k]
        else:
            kv = _median_term(D[:, i] * g)
            v[i] -= Dl[kv, i] * gl[kv]
        rho = 1 / (gl @ sl)
        cc = rho * rho * (gl @ (Dl @ gl)) + rho
        bad = Dl - rho * np.outer(sl, v) - rho * np.outer(u, sl) + cc * np.outer(sl, sl)
        assert not R.within(bad.astype(np.float64), ref, bar), which


# ---- every launcher branch is reached by some GPU case ---------------------------------------------------------------------------

def test_gpu_cases_reach_every_launcher_branch():
    mv = {R.matvec_path(n, a, b) for n, a, b in T.MATVEC_CASES}
    assert mv == {"v4", "scalar"}
    assert any(n % 4 == 0 and R.matvec_path(n, a, 0) == "scalar" for n, a, _ in T.MATVEC_CASES)     # by D's alignment
    assert any(n % 4 == 0 and R.matvec_path(n, 0, b) == "scalar" for n, _, b in T.MATVEC_CASES)     # by g's alignment
    assert {R.hinv_rank2_path(n, a, b, c) for n, k, sg, a, b, c in T.HINV_CASES} == {"v4", "double2", "scalar"}
    by_off = {(a, b, c): R.hinv_rank2_path(256, a, b, c) for *_, a, b, c in T.HINV_CASES if (a, b, c) != (0, 0, 0)}
    assert by_off == {(8, 0, 0): "scalar", (16, 0, 0): "double2", (0, 8, 0): "double2", (0, 0, 8): "double2"}
    assert {n % 4 for n, *_ in T.HINV_CASES} == {0, 1, 2, 3}
    assert {k for _, k, *_ in T.HINV_CASES} == {0, 1, 2, 3} and {sg for _, _, sg, *_ in T.HINV_CASES} == {-1, 1}
    # ragged 256-column and 1024-column chunks, one and several row blocks of the v4 pass 1
    v4n = [n for n, k, sg, a, b, c in T.HINV_CASES if R.hinv_rank2_path(n, a, b, c) == "v4"]
    assert any(n % 256 for n in v4n) and any(n % 1024 and n > 1024 for n in v4n)
    assert {R.hinv_v4_blocks(n, 148)[0] == 1 for n in v4n} == {True, False}
    # the literal form's GEMMs take <false> through D's misalignment (D at +8)
    assert any(R.gemm_path(n, n, n, a, a, 0) == "scalar" and n % 2 == 0 for n, k, sg, a, b, c in T.HINV_CASES)
    gp = {R.gemm_path(*c) for c in T.GEMM_CASES}
    assert gp == {"vec16", "scalar"}
    for pos in range(3):
        assert any(N % 2 == 0 and K % 2 == 0 and off[pos] == 8 and R.gemm_path(M, N, K, *off) == "scalar"
                   for M, N, K, *off in T.GEMM_CASES)
    sy = {(R.syrk_path(n, wf, oJ, oF), wf) for m, n, oJ, oF, fm in T.SYRK_CASES for wf in fm}
    assert sy == {("ldgsts16", True), ("ldgsts16", False), ("ldgsts8", True), ("ldgsts8", False)}
    assert any(n % 2 == 0 and oJ == 8 for m, n, oJ, oF, fm in T.SYRK_CASES)                          # <false> by J's alignment
    assert any(n % 16 == 0 and oF == 8 and R.syrk_path(n, True, oJ, oF) == "ldgsts16"                # F refused by the TMA
               for m, n, oJ, oF, fm in T.SYRK_CASES)
    nb = max((n + 127) // 128 for m, n, *_ in T.SYRK_CASES)
    assert nb * (nb + 1) // 2 > 148                                                                   # more than one wave
