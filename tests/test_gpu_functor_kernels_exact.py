"""The generic functor kernels of include/pnol/device/functor_kernels.cuh bit for bit, on every path their launchers pick and up to
each launcher's shared-memory limit: the population sweep, the forward-difference gradient (plain and over an active set), the FD
Hessian, the alpha pool, the residual, the black-box FD Jacobian and the analytic Jacobian; and the refusals one past the limits.

References: the oracle (tests/oracle_lib.py) for the built-in objectives; for the residual model of any width n
(tests/user_functor/my_wide_models.hpp, built out of tree by tests/user_wide_lib.py) its own __host__ __device__ code run on the host,
with numpy's IEEE quotient (r_j - r_0) / dx_j for the forward difference. Every result is compared as uint64 bits, so -0 and +0
differ. Device buffers are guarded by 0xFF bands and placed 0, 8, 16 or 24 bytes past 256-byte alignment.

Which kernel each case reaches (restated in exact_reference.py: eval_batch_path, jacobian_tile_rows, max_n; test_functor_kernels_cpu.py
checks on the CPU that every branch is taken by some case below). smem_optin = 232 448 bytes (B200):

  eval_batch (Power, separable)  rowwise16 / rowwise           n % 4 == 0, ld % 4 == 0, rows 32-byte aligned; n % 16 == 0 or not
                                 warp-tile, n == 32            otherwise, B >= 64, 24 <= n <= 113: whole 32-row batches / the last
                                 ("warp32_full" / "_ragged")   partial batch
                                 warp-tile, general n          the same with n != 32
                                 tile16 / tile_scalar          otherwise, n <= 227: ld == n, n even, 16-byte aligned rows or not
                                 direct                        n >= 228
  jacobian (analytic)            128 / 64 / 32 rows a tile     n <= 225 / 447 / 879; untiled from n = 880
  fd_jacobian (black box)        one column pass of 32 per 32 columns, ragged last pass; div_exact's fast quotient, or `/` for a
                                 divisor outside 2^+-200 or with an all-ones significand, or a dividend outside 2^+-700

Rows of the sweep that are left off keep the NaN payload f_out held. A batch larger than one wave (2048 threads an SM bound it for
any occupancy) makes the grid-stride loops run at least twice; so does a row count past one wave of the analytic Jacobian at every
tile size, untiled included (n = 880: 303 233 rows, 2.1 GB of J, compared in chunks of rows).

Refusals: alpha_pool, residual, fd_jacobian and fd_points one past their limits. pnol_fd_hessian runs fd_points first, at the same
8 n bytes, so through the C-ABI its refusal is fd_points' and fd_hessian's own check is not reached.
"""
import ctypes as C

import numpy as np
import pytest

import exact_reference as R
import oracle_lib as O
import user_wide_lib as UW
from parallelnonlinearoptimizationlibrary_b200 import capi
from test_gpu_dense_exact import Buffers

pytestmark = pytest.mark.gpu

OPTIN = R.SMEM_OPTIN_B200
NAN_PAYLOAD = np.array([0x7FF8_0000_DEAD_BEEF], dtype=np.uint64).view(np.float64)[0]
TINY_DIVIDEND_ROW = 17                  # rows i % 17 == 5 of the wide model get t = 2^-760: dividends below 2^-700


# ---- cases ----------------------------------------------------------------------------------------------------------------------

EVAL_GEOMS = [  # (n, ld, offset of the points)
    (32, 32, 0), (64, 64, 0), (320, 324, 0),                           # rowwise16
    (4, 4, 0), (20, 20, 0), (36, 40, 0), (228, 228, 0),                # rowwise
    (32, 32, 8), (32, 33, 0), (32, 32, 16),                            # warp-tile at n == 32 (B < 64: the tile kernel)
    (33, 33, 0), (24, 24, 24), (113, 113, 0), (100, 100, 16),          # warp-tile, general n
    (23, 23, 0), (114, 114, 8), (227, 227, 0),                         # tile, element by element
    (22, 22, 0), (114, 114, 16), (226, 226, 0),                        # tile, 16-byte staging
    (228, 228, 8), (229, 229, 0), (500, 512, 24),                      # direct
]
EVAL_B = [1, 31, 32, 33, 63, 64, 65]
EVAL_WAVE_GEOMS = [(32, 32, 0), (4, 4, 0), (32, 32, 8), (33, 33, 0), (23, 23, 0), (22, 22, 0)]
EVAL_CASES = [g + (B,) for g in EVAL_GEOMS for B in EVAL_B] + [g + ("wave",) for g in EVAL_WAVE_GEOMS]

FDG_N = [1, 31, 32, 33, 255, 256, 257, R.max_n("fd_points", OPTIN)]
FDH_N = [2, 33, 200, 1000]
JAC_N = [1, 31, 32, 33, 63, 64, 65, 100, 1000, R.max_n("fd_jacobian", OPTIN)]
JAC_M = [1, 127, 128, 129]
JAC_CASES = [(n, m) for n in JAC_N for m in JAC_M] + [(n, "wave") for n in JAC_N if n <= 100]
DX_KINDS = ["1e-7", "1e-5", "negative", "1e-70", "all-ones"]
RES_N = [1, 33, 1000, R.max_n("residual", OPTIN)]
AJ_N = [3, 33, 225, 226, 447, 448, 879, 880, 2000]
AJ_CASES = [(n, m) for n in AJ_N for m in (1, 129, 1000)] + [(n, "wave") for n in AJ_N if n <= 880]
AJ_CHUNK_ROWS = 16384                   # rows of J read back and compared at a time


def _id(case):
    return "-".join(str(v) for v in case)


# ---- helpers --------------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def props(ctx):
    """the device properties the launchers read (capi.cu: pnol_ctx_create); the case table is laid out for a B200's opt-in"""
    import torch
    p = torch.cuda.get_device_properties(ctx.device)
    assert p.shared_memory_per_block_optin == OPTIN, p.shared_memory_per_block_optin
    assert p.multi_processor_count == ctx.sm_count
    return p


@pytest.fixture(scope="module")
def wide():
    return UW.build_and_load()


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def _same(got, want, what, nan_any=False):
    """bit for bit; nan_any: a NaN matches a NaN of any payload (the device's and the host's default NaNs differ)"""
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape, what
    ok = _bits(got) == _bits(want)
    if nan_any:
        ok |= np.isnan(got) & np.isnan(want)
    assert ok.all(), "%s: %d of %d entries differ, first at %s: %r vs %r" % (
        what, np.count_nonzero(~ok), ok.size, np.argwhere(~ok)[0], got[~ok][0], want[~ok][0])


def _p(v):
    return C.c_void_p(v)


def _wave_rows(ctx, threads, smem, props):
    """an upper bound on the rows one wave of a grid-stride kernel covers: blocks an SM can hold by threads and by shared memory"""
    per_sm = min(props.max_threads_per_multi_processor // threads, props.shared_memory_per_multiprocessor // max(smem, 1))
    return ctx.sm_count * max(per_sm, 1) * threads


def _mixed_dx(n, rng):
    """mixed sign and size, one 1e-70 step (a zero difference keeps the sign of its step)"""
    dx = rng.choice([1e-7, -1e-6, 3e-5, -2.5e-8, 1e-4], size=n)
    dx[n // 2] = -1e-70
    return dx


# ---- eval_batch -----------------------------------------------------------------------------------------------------------------

def _patterns(B):
    """indicator patterns: none, alternating, one 128-row tile off, one 32-row batch off, the last row only"""
    i = np.arange(B)
    tile = (i >= 128) & (i < 256) if B > 256 else i < 128
    warp = (i >= 32) & (i < 64) if B > 64 else i < 32
    return [("all", None), ("alternating", i % 2 == 0), ("tile-off", ~tile), ("batch-off", ~warp), ("last-only", i == B - 1)]


def _eval_points(B, n, ld, rng):
    """B rows of ld doubles: uniform in [-2, 2], every fifth row an order witness (n >= 3), the padding past n NaN"""
    pts = np.full((B, ld), np.nan)
    pts[:, :n] = rng.uniform(-2.0, 2.0, size=(B, n))
    if n >= 3:
        for k, w in enumerate(R.order_witnesses(n)):
            pts[5 * k::15, :n] = w
    return pts


@pytest.mark.parametrize("case", EVAL_CASES, ids=_id)
def test_eval_batch_separable_bit_exact(ctx, props, case):
    n, ld, off, B = case
    if B == "wave":
        B = ctx.sm_count * props.max_threads_per_multi_processor + 129       # > one wave of any 128-thread-block kernel
    path = R.eval_batch_path(n, ld, off, B, OPTIN)
    rng = np.random.default_rng(1000 + 7 * n + ld + off + B)
    pts = _eval_points(B, n, ld, rng)
    f = ctx.functor(capi.F_POWER, (), (1,))
    want_all = O.eval_batch(O.OFunctor(capi.F_POWER, (), (1,)), pts[:, :n])
    for name, on in _patterns(B):
        prefill = np.full(B, NAN_PAYLOAD)
        with Buffers(ctx) as bufs:
            P = bufs(pts, off)
            I = bufs(on.astype(np.uint8), 8) if on is not None else None
            Fo = bufs(prefill, (off + 8) % 32)
            ctx.eval_batch(f, P.ptr, B, n, ld, I.ptr if I else None, Fo.ptr)
            got = Fo.read(B)
            if on is None:
                _same(P.read((B, ld)), pts, "points", nan_any=True)
        want = want_all if on is None else np.where(on, want_all, prefill)
        _same(got, want, "f (%s, indicator %s)" % ("/".join(sorted(path)), name))
    f.close()


# ---- forward-difference gradient ------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("n", FDG_N)
def test_fd_gradient_bit_exact(ctx, n):
    rng = np.random.default_rng(2000 + n)
    x, dx = rng.uniform(-1.5, 1.5, n), _mixed_dx(n, rng)
    f = ctx.functor(capi.F_ROSENBROCK)
    gw, f0w = O.fd_gradient(O.OFunctor(capi.F_ROSENBROCK), x, dx)
    o = [0, 8, 16, 24]
    with Buffers(ctx) as bufs:
        xb, db, gb = bufs(x, o[n % 4]), bufs(dx, o[(n + 1) % 4]), bufs(nbytes=8 * n, off=o[(n + 2) % 4])
        f0 = C.c_double()
        ctx.check(ctx.lib.pnol_fd_gradient(ctx.h, f.handle, _p(xb.ptr), _p(db.ptr), n, _p(gb.ptr), C.byref(f0)))
        _same(gb.read(n), gw, "g")
        _same(f0.value, f0w, "f0")
        _same(xb.read(n), x, "x")
    f.close()


def _masks(nfull):
    j = np.arange(nfull)
    return {
        "straddle": ((j >= 250) & (j < 262)) | ((j >= 509) & (j < 517)),   # across assemble_recur_kernel's 256-entry chunks
        "every-third": j % 3 == 1,
        "first-chunk": j < 256,
    }


@pytest.mark.parametrize("extra", [0, 7], ids=["nr=free", "nr>free"])
@pytest.mark.parametrize("mask", ["straddle", "every-third", "first-chunk"])
def test_fd_gradient_recur_bit_exact(ctx, mask, extra):
    nfull = 700
    ind = _masks(nfull)[mask]
    nr = int(np.count_nonzero(~ind)) + extra               # extra: more reduced entries than free slots (their stencil is f(x))
    rng = np.random.default_rng(3000 + nr)
    xr, dxr = rng.uniform(-1.5, 1.5, nr), _mixed_dx(nr, rng)
    const_x = rng.uniform(-1.0, 1.0, nfull)
    f = ctx.functor(capi.F_ROSENBROCK)
    g, f0 = ctx.fd_gradient_recur(f, xr, dxr, const_x, ind)
    gw, f0w = O.fd_gradient_recur(O.OFunctor(capi.F_ROSENBROCK), xr, dxr, const_x, ind)
    _same(g, gw, "g (%s)" % mask)
    _same(f0, f0w, "f0")
    f.close()


# ---- forward-difference Hessian -------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("n", FDH_N)
def test_fd_hessian_distinct_steps_bit_exact(ctx, n):
    """a distinct dx_i per coordinate: an entry computed for the wrong pair, or divided by the wrong steps, is seen"""
    rng = np.random.default_rng(4000 + n)
    x = rng.uniform(-1.2, 1.2, n)
    dx = 1e-3 * (1.0 + np.arange(n) / n) * np.where(np.arange(n) % 3 == 2, -1.0, 1.0)
    f = ctx.functor(capi.F_ROSENBROCK)
    Bw = O.fd_hessian(O.OFunctor(capi.F_ROSENBROCK), x, dx)
    with Buffers(ctx) as bufs:
        xb, db, Bb = bufs(x, 8), bufs(dx, 16), bufs(nbytes=8 * n * n, off=24)
        ctx.check(ctx.lib.pnol_fd_hessian(ctx.h, f.handle, _p(xb.ptr), _p(db.ptr), n, _p(Bb.ptr)))
        _same(Bb.read((n, n)), Bw, "B")
    f.close()


# ---- alpha pool -----------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("active_set", [False, True], ids=["plain", "active-set"])
def test_alpha_pool_at_its_limit_bit_exact(ctx, active_set):
    """n = the largest the pool's 17 n + 16 bytes allow; a step of 1e300 overflows f: phi takes the 1e10 sentinel, its slope NaN"""
    nfull = R.max_n("alpha_pool", OPTIN)
    rng = np.random.default_rng(5000 + active_set)
    alpha = np.array([0.0, 1e-3, 0.5, 1.0, 1e300, 2.0, 1e-8])
    eval_ind = np.array([1, 1, 0, 1, 1, 0, 1], dtype=np.uint8)
    kw = {}
    n = nfull
    if active_set:
        ind = _masks(nfull)["straddle"] | (np.arange(nfull) % 5 == 0)
        n = int(np.count_nonzero(~ind))
        kw = dict(const_x=rng.uniform(-1.0, 1.0, nfull), const_ind=ind.astype(np.uint8))
    x, p = rng.uniform(-1.0, 1.0, n), rng.normal(size=n) * 1e-2
    f = ctx.functor(capi.F_ROSENBROCK)
    got = ctx.alpha_pool(f, x, p, alpha, 1e-6, True, eval_ind, **kw)
    want = O.alpha_pool(O.OFunctor(capi.F_ROSENBROCK), x, p, alpha, 1e-6, True, eval_ind, **kw)
    _same(got[0], want[0], "phi")
    _same(got[1], want[1], "dphi", nan_any=True)
    assert got[2] == want[2] == 1
    assert np.isnan(got[1][4]) and got[0][4] == 1e10
    f.close()


# ---- residual and black-box FD Jacobian of the wide model ----------------------------------------------------------------------

def _dx(kind, n, rng):
    if kind == "1e-7":
        return np.full(n, 1e-7)
    if kind == "1e-5":
        return np.full(n, 1e-5)
    if kind == "negative":
        return -1e-6 * (1.0 + np.arange(n) % 7)
    if kind == "1e-70":
        return np.full(n, 1e-70)                       # outside 2^+-200: make_recip gives 0, the quotient is `/` (nonzero
                                                       # dividends only at the coordinates _wide_problem makes tiny)
    return np.full(n, np.nextafter(2.0 ** -20, 0.0))  # all-ones significand: `/`


def _wide_problem(n, m, seed):
    """columns and x of the wide model. Every fifth coordinate of x is of order 1e-62, so that a step of 1e-70 moves it, and the rows
    i % 17 == 11 have s = y = 0, so that their residual keeps that difference: the quotient `/` also sees nonzero dividends"""
    rng = np.random.default_rng(seed)
    cols = UW.columns(m, rng, tiny_rows=np.arange(5, m, TINY_DIVIDEND_ROW), bare_rows=np.arange(11, m, TINY_DIVIDEND_ROW))
    x = rng.uniform(-2.0, 2.0, n)
    x[::5] *= 1e-62
    return cols, x, rng


@pytest.mark.parametrize("case", JAC_CASES, ids=_id)
def test_fd_jacobian_blackbox_bit_exact(ctx, wide, case):
    n, m = case
    if m == "wave":
        m = ctx.sm_count * 4 * 128 + 129                # the kernel's grid is at most 4 blocks of 128 rows an SM
    cols, x, rng = _wide_problem(n, m, 6000 + n + m)
    f = ctx.functor(UW.MYW_F_WIDE, (), (), cols, m)
    o = [0, 8, 16, 24]
    for k, kind in enumerate(DX_KINDS):
        dx = _dx(kind, n, rng)
        Jw, Fw = UW.host_fd_jacobian(cols, x, dx)
        with Buffers(ctx) as bufs:
            xb, db = bufs(x, o[k % 4]), bufs(dx, o[(k + 1) % 4])
            Jb, Fb = bufs(nbytes=8 * m * n, off=o[(k + 2) % 4]), bufs(nbytes=8 * m, off=o[(k + 3) % 4])
            ctx.check(ctx.lib.pnol_fd_jacobian(ctx.h, f.handle, _p(xb.ptr), _p(db.ptr), n, _p(Jb.ptr), _p(Fb.ptr), capi.JAC_BLACKBOX))
            _same(Jb.read((m, n)), Jw, "J (dx %s)" % kind)
            _same(Fb.read(m), Fw, "F (dx %s)" % kind)
    f.close()


@pytest.mark.parametrize("n", RES_N)
def test_residual_bit_exact(ctx, wide, n):
    m = 1000
    cols, x, _ = _wide_problem(n, m, 7000 + n)
    f = ctx.functor(UW.MYW_F_WIDE, (), (), cols, m)
    _, Fw = UW.host_rows(cols, x, want_j=False)
    with Buffers(ctx) as bufs:
        xb, Fb = bufs(x, 8), bufs(nbytes=8 * m, off=16)
        ctx.check(ctx.lib.pnol_residual_eval(ctx.h, f.handle, _p(xb.ptr), n, _p(Fb.ptr), None))
        _same(Fb.read(m), Fw, "F")
    f.close()


# ---- analytic Jacobian of the wide model ----------------------------------------------------------------------------------------

@pytest.mark.parametrize("case", AJ_CASES, ids=_id)
def test_analytic_jacobian_every_tile_size_bit_exact(ctx, wide, props, case):
    n, m = case
    rows = R.jacobian_tile_rows(n, OPTIN)
    if m == "wave":
        threads = rows or 128                          # untiled: 128 threads, only the point in shared memory
        smem = 8 * n + (rows * 8 * (n | 1) if rows else 0)
        m = _wave_rows(ctx, threads, smem, props) + 129
    cols, x, _ = _wide_problem(n, m, 8000 + n + m)
    f = ctx.functor(UW.MYW_F_WIDE, (), (), cols, m)
    with Buffers(ctx) as bufs:
        xb = bufs(x, 24)
        Jb, Fb = bufs(nbytes=8 * m * n, off=8), bufs(nbytes=8 * m, off=16)
        ctx.check(ctx.lib.pnol_fd_jacobian(ctx.h, f.handle, _p(xb.ptr), None, n, _p(Jb.ptr), _p(Fb.ptr), capi.JAC_ANALYTIC))
        for i0 in range(0, m, AJ_CHUNK_ROWS):
            i1 = min(m, i0 + AJ_CHUNK_ROWS)
            Jw, Fw = UW.host_rows(cols, x, True, i0, i1)
            _same(ctx.to_host(Jb.ptr + 8 * i0 * n, (i1 - i0, n)), Jw, "J rows %d.. (%s rows a tile)" % (i0, rows))
            _same(ctx.to_host(Fb.ptr + 8 * i0, i1 - i0), Fw, "F rows %d.." % i0)
    f.close()


# ---- refusals one past each limit -----------------------------------------------------------------------------------------------

def _refused(ctx, call):
    l0 = ctx.launches()
    with pytest.raises(capi.PnolError, match=r"^INVALID"):
        call()
    assert ctx.launches() == l0


def test_refusals_one_past_the_limit_leave_the_context_working(ctx, wide, props):
    """props first: the sizes below are one past the limits of THIS device's opt-in, so an accepted call fails an assertion after a
    few small evaluations rather than running a full-size computation"""
    rng = np.random.default_rng(9000)
    rosen = ctx.functor(capi.F_ROSENBROCK)
    n = R.max_n("alpha_pool", OPTIN) + 1
    _refused(ctx, lambda: ctx.alpha_pool(rosen, np.zeros(n), np.ones(n), np.array([0.0, 1.0]), 1e-6))
    # pnol_fd_hessian runs its stencil points (fd_points, the same 8 n bytes) first. fd_points' refusal is checked on its own
    # through pnol_fd_gradient, whose output is n doubles, before pnol_fd_hessian is called with an output of 8 bytes
    n = R.max_n("fd_hessian", OPTIN) + 1
    assert n == R.max_n("fd_points", OPTIN) + 1
    x, dx = np.zeros(n), np.full(n, 1e-3)
    _refused(ctx, lambda: ctx.fd_gradient(rosen, x, dx))
    with Buffers(ctx) as bufs:
        Bb = bufs(nbytes=8)                            # never written: the call is refused before any launch
        _refused(ctx, lambda: ctx.check(ctx.lib.pnol_fd_hessian(ctx.h, rosen.handle, _p(x.ctypes.data), _p(dx.ctypes.data), n,
                                                                 _p(Bb.ptr))))
    m = 129
    cols, _, _ = _wide_problem(1, m, 9001)
    wf = ctx.functor(UW.MYW_F_WIDE, (), (), cols, m)
    n = R.max_n("residual", OPTIN) + 1
    _refused(ctx, lambda: ctx.residual_eval(wf, np.zeros(n)))
    n = R.max_n("fd_jacobian", OPTIN) + 1
    _refused(ctx, lambda: ctx.fd_jacobian(wf, np.zeros(n), np.full(n, 1e-7), mode=capi.JAC_BLACKBOX))
    # the context still computes
    x = rng.uniform(-1.0, 1.0, 64)
    J, F = ctx.fd_jacobian(wf, x, np.full(64, 1e-7), mode=capi.JAC_BLACKBOX)
    Jw, Fw = UW.host_fd_jacobian(cols, x, np.full(64, 1e-7))
    _same(J, Jw, "J after the refusals")
    _same(F, Fw, "F after the refusals")
    g, f0 = ctx.fd_gradient(rosen, x, np.full(64, 1e-7))
    gw, f0w = O.fd_gradient(O.OFunctor(capi.F_ROSENBROCK), x, np.full(64, 1e-7))
    _same(g, gw, "g after the refusals")
    wf.close()
    rosen.close()
