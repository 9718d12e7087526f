"""TEST INFRASTRUCTURE (CPU only): exact and extended-precision references for the LM linear algebra.

* graded_integer_matrix / periodic_graded_matrix: J = K diag(2^-s) with integer K, |K| <= 2^b and m 4^b < 2^53. Every product
  and every partial sum of J^T J and J^T F (F integer, |F| <= 2^b) is then a multiple of 2^-(s_j + s_l) below 2^53 times it, i.e.
  exactly representable: the result is independent of the summation order, and numpy's float64 BLAS product is exact.
* refined_solution / backward_error: a Cholesky solution refined with residuals in long double (64-bit significand on x86-64),
  and the normwise backward error eta = ||b - A x||_inf / (||A||_inf ||x||_inf + ||b||_inf).
* spd_family: the matrix families of the solve sweep.
"""
import numpy as np
import scipy.linalg

U = 2.0 ** -53                       # unit roundoff of float64
SCALE_MAX = 40                       # column scales 2^-s, s in [0, SCALE_MAX]
PERIOD = 4099                        # periodic rows: odd, so the pattern shifts against every chunk and tile boundary


def integer_bits(m):
    """largest b with m 4^b < 2^53"""
    b = 0
    while m * 4 ** (b + 1) < 2 ** 53:
        b += 1
    return b


class GradedInteger:
    """J = K * 2^-s (column scales), F integer; exact J^T J / J^T F by integer arithmetic."""

    def __init__(self, K, s, F):
        self.K, self.s, self.F = K, s, F
        self.scale = np.ldexp(1.0, -s)                       # 2^-s_j
        self.counts = None                                   # periodic: how often each base row occurs

    @property
    def J(self):
        return self.K.astype(np.float64) * self.scale

    def jtj_int_entry(self, j, l):
        """(K^T K)[j, l] in int64 (exact: below 2^53)"""
        w = self.K[:, j] * self.K[:, l]
        return int(np.dot(self.counts, w)) if self.counts is not None else int(w.sum())

    def jtf_int(self):
        w = self.K * self.F[:, None]
        return (self.counts @ w) if self.counts is not None else w.sum(axis=0)

    def jtj(self):
        """exact J^T J in float64. Through BLAS: exact by the bound (see the module doc; tests/test_exact_reference.py checks it)"""
        Kf = self.K.astype(np.float64)
        G = Kf.T @ (Kf * self.counts[:, None]) if self.counts is not None else Kf.T @ Kf
        return G * np.outer(self.scale, self.scale)

    def jtf(self):
        Kf = self.K.astype(np.float64)
        w = self.F * self.counts if self.counts is not None else self.F
        return (Kf.T @ w.astype(np.float64)) * self.scale


def _scales(n, rng):
    # s_j over [0, 40], permuted: every 128-column tile mixes scales
    return rng.permutation(np.arange(n) % (SCALE_MAX + 1))


def graded_integer_matrix(m, n, rng, zero_rows=3, zero_cols=2):
    """J (m x n) = integers in [-2^b, 2^b] times 2^-s_j, b the largest with m 4^b < 2^53; a few zero rows and columns;
    F integer in [-2^b, 2^b]. Returns a GradedInteger."""
    b = integer_bits(m)
    K = rng.integers(-2 ** b, 2 ** b, size=(m, n), endpoint=True, dtype=np.int64)
    if m > 2:
        K[rng.choice(m, size=min(zero_rows, m - 1), replace=False)] = 0
    if n > 2:
        K[:, rng.choice(n, size=min(zero_cols, n - 1), replace=False)] = 0
    F = rng.integers(-2 ** b, 2 ** b, size=m, endpoint=True, dtype=np.int64)
    return GradedInteger(K, _scales(n, rng), F)


def periodic_graded_matrix(m, n, rng, period=PERIOD):
    """J[i] = base[i mod P] (P = 4099): the exact J^T J is the count-weighted integer product of the P base rows. b is chosen
    for the full m. Returns a GradedInteger whose K / F hold the P base rows and `counts` their multiplicities; J_rows(i0, i1)
    materialises rows [i0, i1)."""
    b = integer_bits(m)
    K = rng.integers(-2 ** b, 2 ** b, size=(period, n), endpoint=True, dtype=np.int64)
    K[rng.choice(period, size=3, replace=False)] = 0
    F = rng.integers(-2 ** b, 2 ** b, size=period, endpoint=True, dtype=np.int64)
    g = GradedInteger(K, _scales(n, rng), F)
    g.m = m
    g.counts = np.full(period, m // period, dtype=np.int64)
    g.counts[:m % period] += 1
    return g


def periodic_rows(g, i0, i1):
    """rows [i0, i1) of the periodic J (float64) and F (float64)"""
    idx = np.arange(i0, i1) % g.K.shape[0]
    return g.K[idx].astype(np.float64) * g.scale, g.F[idx].astype(np.float64)


# ---- solves --------------------------------------------------------------------------------------------------------------------

def residual_ld(A, x, b):
    """b - A x in long double"""
    Al, xl, bl = (np.asarray(v, dtype=np.longdouble) for v in (A, x, b))
    return bl - Al @ xl


def refined_solution(A, b, steps=4):
    """scipy Cholesky in float64 plus `steps` steps of iterative refinement with the residual in long double"""
    c = scipy.linalg.cho_factor(A, lower=True)
    x = scipy.linalg.cho_solve(c, b).astype(np.longdouble)
    bl = np.asarray(b, dtype=np.longdouble)
    Al = np.asarray(A, dtype=np.longdouble)
    for _ in range(steps):
        r = bl - Al @ x
        x = x + scipy.linalg.cho_solve(c, r.astype(np.float64)).astype(np.longdouble)
    return x.astype(np.float64)


def backward_error(A, x, b):
    """eta = ||b - A x||_inf / (||A||_inf ||x||_inf + ||b||_inf), residual in long double"""
    r = residual_ld(A, x, b)
    nA = np.max(np.sum(np.abs(np.asarray(A, dtype=np.longdouble)), axis=1))
    den = nA * np.max(np.abs(np.asarray(x, dtype=np.longdouble))) + np.max(np.abs(np.asarray(b, dtype=np.longdouble)))
    return float(np.max(np.abs(r)) / den)


def forward_error(x, xref, D=None):
    """||x - xref||_inf / ||xref||_inf, in the D-scaled norm ||D .|| when D (a diagonal, as a vector) is given"""
    d = np.ones_like(xref) if D is None else D
    return float(np.max(np.abs(d * (x - xref))) / np.max(np.abs(d * xref)))


def kappa2(A):
    w = np.linalg.eigvalsh(A)
    return float(w[-1] / w[0])


FAMILIES = ("random", "graded", "geometric")


def spd_family(name, n, rng, want_kappa=True):
    """(A, b, D, kappa): A SPD of one family; D the diagonal scaling of the family's natural norm (None: plain), kappa the 2-norm
    condition number that bounds its forward error (of C for the graded family D C D).
      random     M^T M + 0.1 I, M (n + 20) x n normal
      graded     D C D, D = diag(10^linspace(-6, 6)), C a well-conditioned correlation matrix
      geometric  Q diag(geomspace(1, 1e-12)) Q^T, Q random orthogonal"""
    b = rng.normal(size=n)
    if name == "random":
        M = rng.normal(size=(n + 20, n))
        A = M.T @ M + 0.1 * np.eye(n)
        return A, b, None, kappa2(A) if want_kappa else None
    if name == "graded":
        M = rng.normal(size=(2 * n + 20, n))
        S = M.T @ M + n * np.eye(n)
        d = 1.0 / np.sqrt(np.diag(S))
        C = S * np.outer(d, d)
        C = 0.5 * (C + C.T)
        D = 10.0 ** np.linspace(-6, 6, n)
        A = C * np.outer(D, D)
        return A, b, D, kappa2(C) if want_kappa else None
    if name == "geometric":
        Q, _ = np.linalg.qr(rng.normal(size=(n, n)))
        ev = np.geomspace(1.0, 1e-12, n) if n > 1 else np.ones(1)
        A = (Q * ev) @ Q.T
        A = 0.5 * (A + A.T)
        return A, b, None, kappa2(A) if want_kappa else None
    raise ValueError(name)


# LM-like matrices: J^T J of the Lorentz problem at K = n / 2 terms, K a power of two (the sizes the structured Jacobian kernel
# serves; the model's J^T J is positive definite there)
LM_SIZES = (2, 4, 8, 16, 32, 64, 128, 256, 512)
LM_LAMBDAS = (1e-1, 1e-4, 1e-8)


def lm_like(JTJ, lam):
    """A = J^T J with A_ii = (1 + lambda) J^T J_ii (the Marquardt damping, in the kernel's arithmetic)"""
    A = JTJ.copy()
    A[np.diag_indices_from(A)] = (1 + lam) * np.diag(JTJ)
    return A


def ldl_indefinite(n, k, rng, off=0.1):
    """L D L^T with unit lower L (entries off / sqrt(n)) and d_j = 1 except d_k = -1: the Cholesky pivots 0..k-1 are positive and
    pivot k (0-based) is the first non-positive one"""
    L = np.tril(rng.uniform(-1, 1, size=(n, n)) * off / np.sqrt(n), -1) + np.eye(n)
    d = np.ones(n)
    d[k] = -1.0
    return (L * d) @ L.T


def solve_sizes():
    """every n in 1..80, n = -1, 0, 1, 2, 3 mod 32 up to 704, and the edges of the two back-substitution buffer plans"""
    s = set(range(1, 81))
    for q in range(32, 705 + 32, 32):
        s.update(q + r for r in (-1, 0, 1, 2, 3))
    s.update((416, 417, 511, 512, 513, 703, 704))
    return sorted(v for v in s if 1 <= v <= 704)
