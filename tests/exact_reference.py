"""TEST INFRASTRUCTURE (CPU only): exact and extended-precision references for the LM linear algebra.

* graded_integer_matrix / periodic_graded_matrix: J = K diag(2^-s) with integer K, |K| <= 2^b and m 4^b < 2^53. Every product
  and every partial sum of J^T J and J^T F (F integer, |F| <= 2^b) is then a multiple of 2^-(s_j + s_l) below 2^53 times it, i.e.
  exactly representable: the result is independent of the summation order, and numpy's float64 BLAS product is exact.
* refined_solution / backward_error: a Cholesky solution refined with residuals in long double (64-bit significand on x86-64),
  and the normwise backward error eta = ||b - A x||_inf / (||A||_inf ||x||_inf + ||b||_inf).
* spd_family: the matrix families of the solve sweep.
* GradedMatvec / GradedGemm / IntegerHinv: exact inputs and results of p = -D g, C = A B and updateHessianInv; the launchers'
  path predicates restated (matvec_path, hinv_rank2_path, gemm_path, syrk_path); componentwise gamma_d bars against long-double
  references (matvec_bar, gemm_bar, hinv_bar) with each kernel's summation depth.
* eval_batch_path / jacobian_tile_rows / max_n / recip_usable / dividend_in_range: the choices of the generic functor launchers
  (include/pnol/device/functor_kernels.cuh) and of the FD quotient restated; order_witnesses: rows whose sequential sum no other
  summation order reproduces.
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


# ---- the dense BFGS pieces and the DMMA GEMM: exact constructions --------------------------------------------------------------
#
# Every value below is an integer times a power of two, and every product and every partial sum of the kernels' arithmetic is an
# integer multiple of one power of two whose magnitude stays below 2^53 times it. Each is then representable, so the result is
# the exact one in any summation order, fused or not: the kernels must return it bit for bit.

def _exponents(n, lo, hi, rng):
    """n exponents in [lo, hi], each value about equally often, permuted: every 4-wide lane group and 128-column group mixes them"""
    return rng.permutation(np.arange(n) % (hi - lo + 1) + lo).astype(np.int32)


def _zero_some(K, rng, rows=3, cols=2):
    m, n = K.shape
    if m > 2:
        K[rng.choice(m, size=min(rows, m - 1), replace=False)] = 0
    if n > 2:
        K[:, rng.choice(n, size=min(cols, n - 1), replace=False)] = 0


class GradedMatvec:
    """p = -D g with D_ik = K_ik 2^(-r_i - t_k), g_k = G_k 2^(t_k): every product of row i is an integer times 2^(-r_i) and
    n max|K| max|G| < 2^53, so p_i = -(K G)_i 2^(-r_i) exactly."""

    def __init__(self, n, rng):
        b = integer_bits(n)
        self.K = rng.integers(-2 ** b, 2 ** b, size=(n, n), endpoint=True, dtype=np.int64)
        self.G = rng.integers(-2 ** b, 2 ** b, size=n, endpoint=True, dtype=np.int64)
        _zero_some(self.K, rng)
        self.r, self.t = _exponents(n, 0, 30, rng), _exponents(n, -20, 20, rng)
        self.D = np.ldexp(self.K.astype(np.float64), -self.r[:, None] - self.t[None, :])
        self.g = np.ldexp(self.G.astype(np.float64), self.t)
        self.peak = int(np.abs(self.K).max(initial=0)) * int(np.abs(self.G).max(initial=0)) * n   # bound of any partial sum / 2^-r_i
        self.want = np.ldexp(-(self.K @ self.G).astype(np.float64), -self.r)


class GradedGemm:
    """C = A B with A_ik = K_ik 2^(-r_i), B_kj = L_kj 2^(-c_j), K_dim max|K| max|L| < 2^53: C_ij = (K L)_ij 2^(-r_i - c_j) exactly,
    and numpy's float64 product of the integer matrices is exact too (test_exact_reference.py proves it against int64)."""

    def __init__(self, M, N, K, rng):
        b = integer_bits(K)
        self.Ka = rng.integers(-2 ** b, 2 ** b, size=(M, K), endpoint=True, dtype=np.int64)
        self.Lb = rng.integers(-2 ** b, 2 ** b, size=(K, N), endpoint=True, dtype=np.int64)
        _zero_some(self.Ka, rng, rows=2, cols=1)
        _zero_some(self.Lb, rng, rows=1, cols=2)
        self.r, self.c = _exponents(M, 0, 40, rng), _exponents(N, 0, 40, rng)
        self.A = np.ldexp(self.Ka.astype(np.float64), -self.r[:, None])
        self.B = np.ldexp(self.Lb.astype(np.float64), -self.c[None, :])
        self.peak = int(np.abs(self.Ka).max(initial=0)) * int(np.abs(self.Lb).max(initial=0)) * K

    def int_product_f64(self):
        """K L through float64 BLAS (exact by the bound)"""
        return self.Ka.astype(np.float64) @ self.Lb.astype(np.float64)

    def want(self, KL=None):
        KL = self.int_product_f64() if KL is None else KL
        return np.ldexp(np.ldexp(KL, -self.r[:, None]), -self.c[None, :])


class IntegerHinv:
    """updateHessianInv on an integer, nonsymmetric D and integer g, s with g_0 = 1 and s_0 chosen so that g.s = sign 2^k, i.e.
    rho = sign 2^-k exactly. With u = D g, v = D^T g, gamma = g^T D g (int64):
        4^k D_new = 4^k D - sign 2^k (s v^T + u s^T) + (gamma + sign 2^k) s s^T.
    `peak` bounds (as an integer multiple of the finest power of two involved) every product and partial sum of the rank-2 form
    (u, v, g.s, g.u, rho, cc, the per-entry sum) and of the literal form (M1 D, then (M1 D) M2, then + rho s s^T) in any order;
    below 2^53 both forms are exact and equal `want` bit for bit."""

    def __init__(self, n, k, sign, rng, dbits=None, vbits=None, symmetric=False):
        self.n, self.k, self.sign = n, k, sign
        # |D| <= 16, |g|, |s| <= 8; from n = 2048 on |D| <= 8, |g|, |s| <= 4: s_0 absorbs g.s (about sqrt(n) 2^(2 vbits)), and the
        # literal form's bound grows like s_0^2 |g|^T|D||g|
        dbits = (4 if n < 2048 else 3) if dbits is None else dbits
        vbits = (3 if n < 2048 else 2) if vbits is None else vbits
        D = rng.integers(-2 ** dbits, 2 ** dbits, size=(n, n), endpoint=True, dtype=np.int64)
        if symmetric:
            D = D + D.T
        g = rng.integers(-2 ** vbits, 2 ** vbits, size=n, endpoint=True, dtype=np.int64)
        s = rng.integers(-2 ** vbits, 2 ** vbits, size=n, endpoint=True, dtype=np.int64)
        g[0] = 1
        s[0] += sign * 2 ** k - int(g @ s)
        assert int(g @ s) == sign * 2 ** k
        self.Di, self.gi, self.si = D, g, s
        self.D, self.g, self.s = D.astype(np.float64), g.astype(np.float64), s.astype(np.float64)
        self.u, self.v = D @ g, D.T @ g
        self.gamma = int(g @ self.u)
        self.scaled = self.scaled_update(self.u, self.v)
        self.peak = self._peak()
        self.want = np.ldexp(self.scaled.astype(np.float64), -2 * k)

    def scaled_update(self, u, v):
        """4^k D_new in int64 from the given u (row sums) and v (column sums)"""
        k, sg, s = self.k, self.sign, self.si
        return 4 ** k * self.Di - sg * 2 ** k * (np.outer(s, v) + np.outer(u, s)) + (self.gamma + sg * 2 ** k) * np.outer(s, s)

    def swapped(self):
        """the same update with u and v exchanged (a kernel that reads a row partial where it wants a column partial)"""
        return np.ldexp(self.scaled_update(self.v, self.u).astype(np.float64), -2 * self.k)

    def _peak(self):
        k = self.k
        aD, ag, as_ = np.abs(self.Di), np.abs(self.gi), np.abs(self.si)
        au, av = aD @ ag, aD.T @ ag                          # bounds of every partial sum of u, v
        Gam = int(ag @ au)                                   # ... of g.u
        cc = abs(self.gamma + self.sign * 2 ** k)            # 4^k |cc|
        ms = int(as_.max())
        # rank-2 entry: 4^k |D_ij| + 2^k |s_i| |v|_j + 2^k |u|_i |s_j| + 4^k |cc| |s_i| |s_j|, in units of 4^-k
        r2 = 4 ** k * aD + 2 ** k * (np.outer(as_, av) + np.outer(au, as_)) + cc * np.outer(as_, as_)
        # literal: 2^k (M1 D) partial sums <= X = 2^k |D| + |s| (|D|^T |g|)^T; 4^k ((M1 D) M2) <= 2^k X + (X |g|) |s|^T; + 2^k s s^T
        X = 2 ** k * aD + np.outer(as_, av)
        lit = 2 ** k * X + np.outer(X @ ag, as_) + 2 ** k * np.outer(as_, as_)
        return max(int(au.max()), int(av.max()), Gam, int(ag @ as_), cc * ms, int(r2.max()), int(lit.max()),
                   2 ** k + int(np.outer(as_, ag).max()))


# ---- which kernel each launcher picks (restated from csrc/dense.cu and csrc/dmma.cu) -----------------------------------------
# A device pointer is `offset` bytes past a 256-byte-aligned allocation, so its alignment is that of the offset.

def _al(off, b):
    return off % b == 0


def matvec_path(n, off_D=0, off_g=0):
    """launch_matvec_neg"""
    return "v4" if n % 4 == 0 and _al(off_D, 32) and _al(off_g, 32) else "scalar"


def hinv_rank2_path(n, off_D=0, off_g=0, off_s=0):
    """launch_hinv_rank2: the three-launch v4 plan, or the five-launch plan with the double2 or the scalar pass 2"""
    if n % 4 == 0 and _al(off_D, 32) and _al(off_g, 32) and _al(off_s, 32):
        return "v4"
    return "double2" if n % 2 == 0 and _al(off_D, 16) else "scalar"


HINV_LAUNCHES = {"v4": 3, "double2": 5, "scalar": 5, "literal": 5}   # the literal form: dot2, M1/M2, two GEMMs, + rho s s^T


def gemm_path(M, N, K, off_A=0, off_B=0, off_C=0):
    """launch_dgemm_nn: gemm_nn_kernel<true> (16-byte pieces) or <false>"""
    return "vec16" if N % 2 == 0 and K % 2 == 0 and _al(off_A, 16) and _al(off_B, 16) and _al(off_C, 16) else "scalar"


def syrk_path(n, with_f, off_J=0, off_F=0):
    """launch_syrk for m >= 1: the TMA kernels ("tma", "pair"), or the LDGSTS ring syrk_kernel<true> ("ldgsts16") / <false>"""
    vec16 = n % 2 == 0 and _al(off_J, 16)
    tma = vec16 and n % 16 == 0 and (not with_f or _al(off_F, 16))
    if tma:
        return "pair" if (n + 127) // 128 == 2 and not with_f else "tma"
    return "ldgsts16" if vec16 else "ldgsts8"


# ---- which kernel the functor launchers pick (restated from include/pnol/device/functor_kernels.cuh) ----------------------------
# smem_optin is the device's opt-in shared memory per block (pnol_launch_env::smem_optin; 232 448 bytes on a B200).

SMEM_OPTIN_B200 = 232_448
EVAL_BATCH_PATHS = ("rowwise16", "rowwise", "warp32_full", "warp32_ragged", "warp_general", "tile16", "tile_scalar", "direct")


def eval_batch_path(n, ld, off, B, smem_optin, separable=True):
    """eval_batch (:302-325) and SeparableLaunch<F, true>::run (:269-298) for B >= 1: the set of branches the launch runs when
    every row is evaluated. The warp-tile kernel (:136-184) runs "warp32_full" for whole 32-row batches at n == 32 (:152),
    "warp32_ragged" for a last partial batch at n == 32 (:168), "warp_general" otherwise (:170); the tile kernel (:84-121) stages with
    16-byte loads when ld == n, n is even and the rows are 16-byte aligned (:96), else element by element"""
    if separable:
        pitch = n | 1
        smem = 4 * 32 * pitch * 8
        rowwise_ok = n % 4 == 0 and ld % 4 == 0 and _al(off, 32)
        if rowwise_ok:
            return {"rowwise16" if n % 16 == 0 else "rowwise"}
        if not (smem > smem_optin // 2 or B < 64 or n < 24):
            if n != 32:
                return {"warp_general"}
            return ({"warp32_full"} if B >= 32 else set()) | ({"warp32_ragged"} if B % 32 else set())
    if 128 * (n | 1) * 8 <= smem_optin:
        return {"tile16" if ld == n and n % 2 == 0 and _al(off, 16) else "tile_scalar"}
    return {"direct"}


def jacobian_tile_rows(n, smem_optin):
    """jacobian (:818-841): rows per tile, 128, 64 or 32, or None when the kernel runs untiled"""
    xbytes, row_bytes = 8 * n, 8 * (n | 1)
    threads = 128
    while threads > 32 and xbytes + threads * row_bytes > smem_optin:
        threads //= 2
    return threads if xbytes + threads * row_bytes <= smem_optin else None


def max_n(launcher, smem_optin):
    """the largest n each launcher accepts (its PNOL_DEV_REQUIRE on the dynamic shared memory); n + 1 is refused"""
    w = smem_optin // 8
    return {
        "fd_points": w,                                  # :363  8 n
        "gradient": w,                                   # :407  8 n
        "residual": w,                                   # :698  8 n
        "fd_hessian": w,                                 # :467  8 n
        "hessian": w - 32 * 33,                          # :539  8 (32 * 33 + n)
        "alpha_pool": (smem_optin - 16) // 17,           # :601  17 n + 16
        "alpha_slope": w // 2,                           # :668  8 (nfull + n), n = nfull
        "fd_jacobian": (w - 128 * 33) // 3,              # :766  8 (3 n + 128 * 33)
    }[launcher]


def recip_usable(d):
    """make_recip (include/pnol/device/exact_div.cuh:20-30) gives r = RN(1/d) != 0: |d| within 2^+-200, significand not all ones"""
    b = int(np.array([d], dtype=np.float64).view(np.uint64)[0])
    e = (b >> 52) & 0x7FF
    return 1023 - 200 < e < 1023 + 200 and (b & (2 ** 52 - 1)) != 2 ** 52 - 1


def dividend_in_range(x):
    """div_exact (exact_div.cuh:52-65) takes its FMA sequence for a dividend within 2^+-700, or zero; `/` otherwise"""
    b = int(np.array([x], dtype=np.float64).view(np.uint64)[0])
    e = (b >> 52) & 0x7FF
    return 1023 - 700 < e < 1023 + 700 or x == 0.0


def order_witnesses(n):
    """three rows whose sequential sum from 0 (Power with power 1: the terms are the entries) no other order reproduces, n >= 3:
    [1, e, e, ...] sums to 1, [e, ..., e, 1] to 1 + (n - 1) e rounded once, [1, e, -1, e, ...] to (n - 3) e (e = 2^-53). An order
    that adds two small entries before it meets the 1, or lets the 1 absorb a different set of them (pairwise, reversed, strided,
    four at a time), changes at least one of the three sums (test_functor_kernels_cpu.py)"""
    w = np.full((3, n), U)
    w[0, 0] = w[1, n - 1] = w[2, 0] = 1.0
    w[2, 2] = -1.0
    return w


def seq_sum(v):
    s = 0.0
    for t in v:
        s = s + float(t)
    return s


# ---- componentwise bars on real-valued data ------------------------------------------------------------------------------------

UL = 2.0 ** -64                      # unit roundoff of the x86-64 long double (64-bit significand)


def gamma(d, u=U):
    """gamma_d = d u / (1 - d u): a sum whose terms each pass through at most d roundings is off by at most gamma_d sum |terms|"""
    return d * u / (1 - d * u)


def ld(a):
    return np.asarray(a, dtype=np.longdouble)


def matvec_depth(n, path):
    """roundings a product of p = -D g passes through. v4: a chain of ceil(n / 128) FMA per lane and component, two adds for the
    four components, five butterfly adds; scalar: ceil(n / 32) FMA per lane and five butterfly adds (-1 x: exact)"""
    return -(-n // 128) + 7 if path == "v4" else -(-n // 32) + 5


def gemm_depth(K):
    """roundings a product of C = A B passes through in gemm_nn_kernel: one m8n8k4 DMMA per 4 k, each at most a rounded product
    and four rounded adds into the accumulator for its own terms, four adds for the accumulator it carries"""
    return 4 * (-(-K // 4)) + 1


def hinv_v4_blocks(n, sm_count):
    """(row blocks, rows per block R, column blocks) of hinv_pass1_v4_kernel, restated from launch_hinv_rank2"""
    ncb = -(-n // 256)
    wave = 2 * sm_count
    nrb = (n + 111) // 112
    waves = (nrb * ncb + wave // 2) // wave
    if waves >= 1:
        nrb = waves * wave // ncb
    nrb = max(nrb, 1)
    R = (-(-n // nrb) + 3) & ~3
    return -(-n // R), R, ncb


def hinv_depths(n, path, sm_count):
    """(d_u, d_v, d_dot): roundings a term of u = D g, of v = D^T g and of the dot products g.s, g.u passes through"""
    if path == "v4":
        nrb, R, ncb = hinv_v4_blocks(n, sm_count)
        d_u = 2 + 2 + 5 + -(-ncb // 8) + 8              # 2 FMA per chain, 2 adds, 5 butterfly adds, finish: chain + 8 group adds
        d_v = 4 * -(-R // 32) + 8 + -(-nrb // 8) + 8     # FMA over the warp's rows, 8 warp adds, finish
        d_dot = -(-n // 256) + 8                         # 256-thread chains and an 8-level tree
    else:
        nrb, ncb = -(-n // 32), -(-n // 512)
        d_u = min(16, -(-n // 32)) + 5 + ncb             # chain over the 512-column block, butterfly, finish over column blocks
        d_v = 4 + 8 + nrb                                # 4 rows per warp, 8 warp adds, finish over row blocks
        d_dot = -(-n // 1024) + 10                       # dot2_kernel: 1024-thread chains and a 10-level tree
    return d_u, d_v, d_dot


def hinv_reference_ld(D, g, s):
    """the rank-2 update in long double: (D_new, magnitude terms T = |D| + |rho||s|(|D|^T|g|)^T + |rho|(|D||g|)|s|^T
    + (rho^2 |g|^T|D||g| + |rho|) |s||s|^T, condition of g.s = |g|^T|s| / |g.s|)"""
    Dl, gl, sl = ld(D), ld(g), ld(s)
    u, v = Dl @ gl, Dl.T @ gl
    gs = gl @ sl
    rho = 1 / gs
    cc = rho * rho * (gl @ u) + rho
    want = Dl - rho * np.outer(sl, v) - rho * np.outer(u, sl) + cc * np.outer(sl, sl)
    aD, ag, as_ = np.abs(Dl), np.abs(gl), np.abs(sl)
    au, av = aD @ ag, aD.T @ ag
    T = aD + abs(rho) * (np.outer(as_, av) + np.outer(au, as_)) + (rho * rho * (ag @ au) + abs(rho)) * np.outer(as_, as_)
    return want, T, (ag @ as_) / abs(gs)


def hinv_bar(n, T, kappa_gs, d_u, d_v, d_dot):
    """|D_hat - D_ld| <= (gamma_d + 2 eps_rho) T + (the same for the long-double reference), d = max(d_u, d_v) + d_dot + 8.
    Derivation (first order in u): the computed v_j is off by gamma_{d_v} (|D|^T|g|)_j, u_i by gamma_{d_u} (|D||g|)_i, g.u by
    (gamma_{d_u} + gamma_{d_dot}) |g|^T|D||g|; rho = RN(1 / g.s_hat) by eps_rho = (u + eta) / (1 - eta), eta = gamma_{d_dot} kappa_gs
    relative. rho s_i v_j then carries eps_rho + 2 u + gamma_{d_v}, rho u_i s_j eps_rho + 2 u + gamma_{d_u}, cc s_i s_j (cc = rho^2 g.u
    + rho: one product rounding, rho^2 doubles eps_rho, one add, two products with s) 2 eps_rho + 5 u + gamma_{d_u} + gamma_{d_dot},
    and the sum D + (three terms) adds at most three roundings to each term. gamma_a + gamma_b <= gamma_{a+b} gathers all of it
    under one gamma_d."""
    def part(d_u, d_v, d_dot, u):
        eta = gamma(d_dot, u) * kappa_gs
        eps_rho = (u + eta) / (1 - eta)
        return (gamma(max(d_u, d_v) + d_dot + 8, u) + 2 * eps_rho) * T
    return part(d_u, d_v, d_dot, U) + part(n + 1, n + 1, n + 1, UL)


def matvec_bar(D, g, d):
    """(p in long double, bar): |p_hat - p| <= gamma_d (|D||g|)_i for the kernel's depth d, plus gamma_{n+1} in long double for
    the reference's own error"""
    n = g.size
    return -(ld(D) @ ld(g)), (gamma(d) + gamma(n + 1, UL)) * (np.abs(ld(D)) @ np.abs(ld(g)))


def gemm_bar(A, B, d):
    """(C in long double, bar): gamma_d (|A||B|)_ij plus the long-double reference's gamma_{K+1}"""
    K = A.shape[1]
    return ld(A) @ ld(B), (gamma(d) + gamma(K + 1, UL)) * (np.abs(ld(A)) @ np.abs(ld(B)))


def within(got, ref, bar):
    """componentwise |got - ref| <= bar (in long double); NaN fails"""
    return bool(np.all(np.abs(ld(got) - ref) <= bar))


def graded_scaling(n):
    """10^linspace(-6, 6): the spread of an LM-like inverse Hessian's diagonal"""
    return 10.0 ** np.linspace(-6, 6, n)
