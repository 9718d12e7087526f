"""The checker of tests/test_gpu_lm_linear_algebra.py, checked on the CPU: the integer construction makes numpy's float64 J^T J /
J^T F exact (equal to integer arithmetic bit for bit), an exact comparison notices what the old norm-wise 1e-12 bar does not, and the
solve's bars (backward error eta <= n u, tests/exact_reference.py) are met by scipy's own solution and missed by small perturbations."""
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
