"""The dense FP64 pieces of the BFGS family and the non-TMA SYRK against exact references (tests/exact_reference.py): p = -D g,
both inverse-Hessian updates, the DMMA GEMM and the LDGSTS SYRK bit for bit on integer-times-power-of-two inputs, on every path
their launchers pick; componentwise error bars on real-valued data; the same bits on repeat.

Which kernel each case reaches (restated from the launchers in exact_reference.py; test_exact_reference.py checks on the CPU
that every branch is taken by some case below). Pointers are `offset` bytes past a 256-byte-aligned allocation.

  launcher             branch (restatement)                           taken when                                  reached by
  launch_matvec_neg    matvec_v4_kernel ("v4")                        n % 4 == 0, D and g 32-byte aligned         n % 4 == 0
                       matvec_kernel ("scalar")                       otherwise                                   n % 4 != 0; D or g at +8
  launch_hinv_rank2    pass1_v4, finish_v4, pass2_v4 ("v4", 3)        n % 4 == 0, D, g, s 32-byte aligned         n % 4 == 0
                       pass1, finish x2, dot2, pass2 ("double2", 5)   otherwise, n even, D 16-byte aligned        n % 4 == 2; D at +16; g or s at +8
                       ... with pass2_scalar ("scalar", 5)            otherwise                                   odd n; D at +8
  launch_hinv_literal  dot2, build_m, dgemm x2, add_m3 ("literal", 5) mode HINV_LITERAL                           every update case
  launch_dgemm_nn      gemm_nn_kernel<true> ("vec16")                 N, K even, A, B, C 16-byte aligned          even N and K
                       gemm_nn_kernel<false> ("scalar")               otherwise                                   odd N or K; A, B or C at +8; literal D at +8
  launch_syrk          syrk_kernel<true> ("ldgsts16")                 n even, J 16-byte aligned, not TMA:         n % 16 != 0 even; F at +8
                                                                      n % 16 != 0 or F not 16-byte aligned
                       syrk_kernel<false> ("ldgsts8")                 n odd or J not 16-byte aligned              odd n; J at +8
(the number after a rank-2 plan is its launch count, asserted through ctx.launches())
"""
import ctypes as C

import numpy as np
import pytest

import exact_reference as R
from parallelnonlinearoptimizationlibrary_b200 import capi
from test_gpu_lm_linear_algebra import _check_normal_eq

pytestmark = pytest.mark.gpu

GUARD = 256                          # bytes of 0xFF on either side of every buffer


# ---- cases ----------------------------------------------------------------------------------------------------------------------

MATVEC_N = [1, 2, 3, 4, 5, 8, 127, 128, 129, 508, 512, 516, 1020, 4096, 4100]     # +-4 around 128 kMvUnroll = 512
MATVEC_CASES = [(n, 0, 0) for n in MATVEC_N] + [(512, 8, 0), (512, 0, 8), (4096, 8, 0), (4096, 0, 8)]   # (n, off_D, off_g)

HINV_N = [1, 2, 3, 4, 6, 8, 124, 128, 130, 252, 256, 258, 260, 511, 512, 1022, 1023, 1024, 1028, 4096]
# (n, k, sign, off_D, off_g, off_s): g.s = sign 2^k, k = 0 ... 3 and both signs spread over the sizes
HINV_CASES = [(n, i % 4, -1 if i % 3 == 1 else 1, 0, 0, 0) for i, n in enumerate(HINV_N)] + \
             [(n, 1 + j % 3, -1 if j == 2 else 1) + off for n in (256, 1024)
              for j, off in enumerate([(8, 0, 0), (16, 0, 0), (0, 8, 0), (0, 0, 8)])]

GEMM_M, GEMM_N, GEMM_K = (1, 127, 128, 129, 300), (1, 2, 127, 128, 130, 257), (1, 2, 31, 32, 33, 65, 512)
# (M, N, K, off_A, off_B, off_C): the full product, the even-N, even-K shapes again with one operand at +8, and 4096^3 once
GEMM_CASES = [(M, N, K, 0, 0, 0) for M in GEMM_M for N in GEMM_N for K in GEMM_K] + \
             [(M, N, K) + off for M in (127, 300) for N in GEMM_N if N % 2 == 0 for K in GEMM_K if K % 2 == 0
              for off in [(8, 0, 0), (0, 8, 0), (0, 0, 8)]]
GEMM_BIG = (4096, 4096, 4096)

SYRK_N = [1, 3, 17, 127, 129, 130, 255, 257, 300, 383, 1001, 2500]     # n = 2500: 210 tile roles, more than one wave of CTAs
SYRK_M = [1, 31, 32, 33, 4099, 100_000]
# (m, n, off_J, off_F, with F and / or without); m = 100 000 up to n = 383 (the host reference is m n^2)
SYRK_CASES = [(m, n, 0, 0, (True, False)) for n in SYRK_N for m in SYRK_M if m < 100_000 or n <= 383] + \
             [(m, n, 8, 0, (True, False)) for n in (256, 512) for m in (33, 4099)] + \
             [(m, n, 0, 8, (True,)) for n in (256, 512) for m in (33, 4099)]


def _id(case):
    return "-".join(str(v) for v in case if not isinstance(v, tuple))


# ---- guarded device buffers -----------------------------------------------------------------------------------------------------

class Guarded:
    """GUARD + off bytes of 0xFF, the data (nbytes, starting `off` bytes past 256-byte alignment), GUARD bytes of 0xFF"""

    def __init__(self, ctx, nbytes, off=0, data=None):
        self.ctx, self.nbytes, self.off = ctx, nbytes, off
        self.total = GUARD + off + nbytes + GUARD
        self.base = ctx.malloc(self.total)
        ctx.check(ctx.lib.pnol_memset(ctx.h, C.c_void_p(self.base), 0xFF, C.c_size_t(self.total)))
        self.ptr = self.base + GUARD + off
        if data is not None:
            assert data.nbytes == nbytes
            ctx.memcpy(self.ptr, np.ascontiguousarray(data), nbytes)

    def read(self, shape):
        return self.ctx.to_host(self.ptr, shape)

    def guards_intact(self):
        lo = self.ctx.to_host(self.base, GUARD + self.off, dtype=np.uint8)
        hi = self.ctx.to_host(self.ptr + self.nbytes, GUARD, dtype=np.uint8)
        return bool(np.all(lo == 0xFF) and np.all(hi == 0xFF))

    def free(self):
        self.ctx.free(self.base)


class Buffers:
    """the guarded buffers of one call; checks every guard band on exit"""

    def __init__(self, ctx):
        self.ctx, self.bufs = ctx, []

    def __call__(self, arr=None, off=0, nbytes=None):
        b = Guarded(self.ctx, arr.nbytes if arr is not None else nbytes, off, arr)
        self.bufs.append(b)
        return b

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        try:
            if exc[0] is None:
                bad = [i for i, b in enumerate(self.bufs) if not b.guards_intact()]
                assert not bad, "guard bands overwritten around buffer(s) %s" % bad
        finally:
            for b in self.bufs:
                b.free()


def _same(got, want, what):
    assert np.array_equal(got, want), "%s: %d entries differ" % (what, np.count_nonzero(~(got == want)))


# ---- p = -D g -------------------------------------------------------------------------------------------------------------------

def _matvec(ctx, bufs, D, g, n, off_D=0, off_g=0):
    Db, gb, pb = bufs(D, off_D), bufs(g, off_g), bufs(nbytes=n * 8)
    ctx.matvec_neg(Db.ptr, gb.ptr, n, pb.ptr)
    return pb.read(n), Db, gb


@pytest.mark.parametrize("case", MATVEC_CASES, ids=_id)
def test_matvec_neg_bit_exact(ctx, case):
    n, off_D, off_g = case
    c = R.GradedMatvec(n, np.random.default_rng(100 + n + off_D + 2 * off_g))
    assert c.peak < 2 ** 53
    with Buffers(ctx) as bufs:
        p, Db, gb = _matvec(ctx, bufs, c.D, c.g, n, off_D, off_g)
        _same(p, c.want, "p (%s path)" % R.matvec_path(n, off_D, off_g))
        _same(Db.read((n, n)), c.D, "D")
        _same(gb.read(n), c.g, "g")


# ---- updateHessianInv -----------------------------------------------------------------------------------------------------------

def _hinv(ctx, bufs, D, g, s, n, mode, off_D=0, off_g=0, off_s=0):
    """(D_new, launches, g and s read back)"""
    Db, gb, sb = bufs(D, off_D), bufs(g, off_g), bufs(s, off_s)
    l0 = ctx.launches()
    ctx.bfgs_update_hinv(Db.ptr, gb.ptr, sb.ptr, n, mode)
    launches = ctx.launches() - l0
    return Db.read((n, n)), launches, gb.read(n), sb.read(n)


@pytest.mark.parametrize("case", HINV_CASES, ids=_id)
def test_update_hinv_bit_exact_both_modes(ctx, case):
    n, k, sign, off_D, off_g, off_s = case
    c = R.IntegerHinv(n, k, sign, np.random.default_rng(200 + n + off_D + 2 * off_g + 3 * off_s))
    assert c.peak < 2 ** 53
    path = R.hinv_rank2_path(n, off_D, off_g, off_s)
    for mode, plan in ((capi.HINV_RANK2, path), (capi.HINV_LITERAL, "literal")):
        with Buffers(ctx) as bufs:
            Dn, launches, g, s = _hinv(ctx, bufs, c.D, c.g, c.s, n, mode, off_D, off_g, off_s)
            _same(Dn, c.want, "D_new (%s)" % plan)
            assert launches == R.HINV_LAUNCHES[plan], (plan, launches)
            _same(g, c.g, "g")
            _same(s, c.s, "s")


# ---- C = A B --------------------------------------------------------------------------------------------------------------------

def _gemm(ctx, bufs, A, B, M, N, K, off_A=0, off_B=0, off_C=0):
    Ab, Bb, Cb = bufs(A, off_A), bufs(B, off_B), bufs(nbytes=M * N * 8, off=off_C)
    ctx.dgemm_nn(Ab.ptr, Bb.ptr, Cb.ptr, M, N, K)
    return Cb.read((M, N)), Ab, Bb


def _gemm_exact(ctx, case, seed):
    M, N, K, off_A, off_B, off_C = case
    c = R.GradedGemm(M, N, K, np.random.default_rng(seed))
    assert c.peak < 2 ** 53
    with Buffers(ctx) as bufs:
        Cm, Ab, Bb = _gemm(ctx, bufs, c.A, c.B, M, N, K, off_A, off_B, off_C)
        _same(Cm, c.want(), "C (%s path)" % R.gemm_path(M, N, K, off_A, off_B, off_C))
        _same(Ab.read((M, K)), c.A, "A")
        _same(Bb.read((K, N)), c.B, "B")


@pytest.mark.parametrize("case", GEMM_CASES, ids=_id)
def test_dgemm_nn_bit_exact(ctx, case):
    _gemm_exact(ctx, case, 300 + sum(case))


def test_dgemm_nn_bit_exact_4096(ctx):
    _gemm_exact(ctx, GEMM_BIG + (0, 0, 0), 4096)


# ---- J^T J / J^T F through the LDGSTS SYRK --------------------------------------------------------------------------------------

@pytest.mark.parametrize("case", SYRK_CASES, ids=_id)
def test_normal_eq_ldgsts_syrk_bit_exact(ctx, case):
    m, n, off_J, off_F, f_modes = case
    assert all(R.syrk_path(n, wf, off_J, off_F) in ("ldgsts16", "ldgsts8") for wf in f_modes)
    g = R.graded_integer_matrix(m, n, np.random.default_rng(11 * m + n + off_J + 2 * off_F))
    lam = 0.25
    J, F = g.J, g.F.astype(np.float64)
    JTJw, rhsw = g.jtj(), -g.jtf()
    for with_f in f_modes:
        with Buffers(ctx) as bufs:
            Jb, Fb = bufs(J, off_J), bufs(F, off_F)
            outs = [bufs(nbytes=n * n * 8), bufs(nbytes=n * n * 8), bufs(nbytes=n * 8)]
            ctx.lm_normal_eq(Jb.ptr, Fb.ptr if with_f else None, m, n, lam, JTJ=outs[0].ptr, A=outs[1].ptr, rhs=outs[2].ptr)
            got = [outs[0].read((n, n)), outs[1].read((n, n)), outs[2].read(n)]
            _check_normal_eq(*got, JTJw, rhsw if with_f else np.zeros(n), lam)
            _same(Jb.read((m, n)), J, "J")
            _same(Fb.read(m), F, "F")


# ---- componentwise bars on real-valued data -------------------------------------------------------------------------------------

def _graded(M):
    """M scaled by 10^linspace(-6, 6) on both sides (an LM-like inverse Hessian's spread)"""
    c = R.graded_scaling(M.shape[0])
    return M * np.outer(c, c)


@pytest.mark.parametrize("graded", [False, True], ids=["normal", "graded"])
@pytest.mark.parametrize("n,off_D", [(5, 0), (129, 0), (512, 0), (4096, 0), (4098, 0), (4096, 8)])
def test_matvec_neg_componentwise_bar(ctx, n, off_D, graded):
    """|p_hat - p|_i <= gamma_d (|D||g|)_i, d the roundings a product passes through on the chosen path (R.matvec_depth), plus
    the long-double reference's own gamma_{n+1}"""
    rng = np.random.default_rng(400 + n)
    D = rng.normal(size=(n, n))
    D = _graded(D) if graded else D
    g = rng.normal(size=n)
    path = R.matvec_path(n, off_D)
    ref, bar = R.matvec_bar(D, g, R.matvec_depth(n, path))
    with Buffers(ctx) as bufs:
        p, _, _ = _matvec(ctx, bufs, D, g, n, off_D)
    assert R.within(p, ref, bar), path


@pytest.mark.parametrize("graded", [False, True], ids=["normal", "graded"])
@pytest.mark.parametrize("M,N,K,off_A", [(129, 127, 65, 0), (300, 257, 512, 0), (128, 130, 4096, 0), (300, 130, 512, 8)])
def test_dgemm_nn_componentwise_bar(ctx, M, N, K, off_A, graded):
    """|C_hat - C|_ij <= gamma_d (|A||B|)_ij, d = R.gemm_depth(K) (M N K <= 2^28: the long-double product stays affordable)"""
    assert M * N * K <= 2 ** 28
    rng = np.random.default_rng(500 + M + N + K)
    A, B = rng.normal(size=(M, K)), rng.normal(size=(K, N))
    if graded:
        A = A * R.graded_scaling(M)[:, None]
        B = B * R.graded_scaling(N)[None, :]
    ref, bar = R.gemm_bar(A, B, R.gemm_depth(K))
    with Buffers(ctx) as bufs:
        Cm, _, _ = _gemm(ctx, bufs, A, B, M, N, K, off_A)
    assert R.within(Cm, ref, bar), R.gemm_path(M, N, K, off_A)


def _hinv_real(n, graded, rng):
    D = rng.normal(size=(n, n))
    D = _graded(D) if graded else D
    g = rng.normal(size=n)
    s = 0.1 * g + 0.05 * rng.normal(size=n)
    return D, g, s


@pytest.mark.parametrize("graded", [False, True], ids=["normal", "graded"])
@pytest.mark.parametrize("n,off_D", [(6, 0), (130, 0), (256, 0), (1023, 0), (1024, 0), (1024, 16), (4096, 0)])
def test_update_hinv_rank2_componentwise_bar(ctx, n, off_D, graded):
    """|D_hat - D_new|_ij <= (gamma_d + 2 eps_rho) (|D_ij| + |rho||s_i|(|D|^T|g|)_j + |rho|(|D||g|)_i|s_j|
    + (rho^2 |g|^T|D||g| + |rho|)|s_i s_j|), derived in R.hinv_bar from the depths of the chosen path (R.hinv_depths)"""
    rng = np.random.default_rng(600 + n)
    D, g, s = _hinv_real(n, graded, rng)
    path = R.hinv_rank2_path(n, off_D)
    ref, T, kappa = R.hinv_reference_ld(D, g, s)
    bar = R.hinv_bar(n, T, kappa, *R.hinv_depths(n, path, ctx.sm_count))
    with Buffers(ctx) as bufs:
        Dn, launches, _, _ = _hinv(ctx, bufs, D, g, s, n, capi.HINV_RANK2, off_D)
    assert launches == R.HINV_LAUNCHES[path]
    assert R.within(Dn, ref, bar), path


# ---- the same bits on repeat, on every path -------------------------------------------------------------------------------------

@pytest.mark.parametrize("n,off", [(4096, 0), (4096, 8), (1023, 0)])
def test_matvec_neg_deterministic(ctx, n, off):
    rng = np.random.default_rng(700 + n)
    D, g = rng.normal(size=(n, n)), rng.normal(size=n)
    with Buffers(ctx) as bufs:
        a, _, _ = _matvec(ctx, bufs, D, g, n, off)
        b, _, _ = _matvec(ctx, bufs, D, g, n, off)
    assert np.array_equal(a, b)


@pytest.mark.parametrize("n,off_D,mode", [(1024, 0, capi.HINV_RANK2), (1024, 16, capi.HINV_RANK2), (1024, 8, capi.HINV_RANK2),
                                          (1023, 0, capi.HINV_RANK2), (1024, 8, capi.HINV_LITERAL), (1024, 0, capi.HINV_LITERAL)])
def test_update_hinv_deterministic(ctx, n, off_D, mode):
    D, g, s = _hinv_real(n, False, np.random.default_rng(800 + n))
    with Buffers(ctx) as bufs:
        a = _hinv(ctx, bufs, D, g, s, n, mode, off_D)[0]
        b = _hinv(ctx, bufs, D, g, s, n, mode, off_D)[0]
    assert np.array_equal(a, b)


@pytest.mark.parametrize("M,N,K,off_A", [(300, 258, 512, 0), (300, 258, 512, 8), (300, 257, 65, 0)])
def test_dgemm_nn_deterministic(ctx, M, N, K, off_A):
    rng = np.random.default_rng(900 + M + N + K)
    A, B = rng.normal(size=(M, K)), rng.normal(size=(K, N))
    with Buffers(ctx) as bufs:
        a, _, _ = _gemm(ctx, bufs, A, B, M, N, K, off_A)
        b, _, _ = _gemm(ctx, bufs, A, B, M, N, K, off_A)
    assert np.array_equal(a, b)


@pytest.mark.parametrize("m,n,off_J", [(100_000, 300, 0), (4099, 2500, 0), (100_000, 256, 8)])
def test_normal_eq_ldgsts_syrk_deterministic(ctx, m, n, off_J):
    rng = np.random.default_rng(1000 + n)
    J, F = rng.normal(size=(m, n)), rng.normal(size=m)
    outs = []
    with Buffers(ctx) as bufs:
        Jb, Fb = bufs(J, off_J), bufs(F)
        for _ in range(2):
            o = [bufs(nbytes=n * n * 8), bufs(nbytes=n * n * 8), bufs(nbytes=n * 8)]
            ctx.lm_normal_eq(Jb.ptr, Fb.ptr, m, n, 0.5, JTJ=o[0].ptr, A=o[1].ptr, rhs=o[2].ptr)
            outs.append([o[0].read((n, n)), o[1].read((n, n)), o[2].read(n)])
    assert all(np.array_equal(a, b) for a, b in zip(*outs))
