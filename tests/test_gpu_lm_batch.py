"""Batched Levenberg-Marquardt on the GPU (pnol_lm_batch, LevMarqBatch): every problem of a batch bit for bit oracle_lib.lm on that
problem alone (X, chi^2, lambda, iterations, stopped, F_out against FOpt) for the three built-in models and the user models of
tests/user_functor/my_jacobians.*, the analytic mode against a Python restatement over oracle_lib.lm_normal_eq / lu_solve with J from
the host jacobian(); independence from B, position and neighbours; random samples at 2^20 and 65 536 problems; host / device / misaligned
pointers and the refusals; the plugin class; and a batch split over two GPUs."""
import numpy as np
import pytest

import lm_batch_cases as LC
from parallelnonlinearoptimizationlibrary_b200 import capi

pytestmark = pytest.mark.gpu

PRM = dict(lambda0=1e-3, factor=10.0, dx=1e-7, maxiter=30, xmindiff=1e-9)


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    yield c
    c.close()


def _same(a, b):
    return np.array_equal(np.asarray(a, dtype=np.float64).view(np.uint64), np.asarray(b, dtype=np.float64).view(np.uint64))


def run(ctx, case, kind=None, jac_mode=capi.JAC_AUTO, X=None, **kw):
    prm = dict(PRM, **kw)
    f = ctx.functor(case["kind"] if kind is None else kind, case["scalars"], (), case["columns"], case["columns"][0].size)
    n = case["n"]
    Xv = np.array(case["X0"] if X is None else X, dtype=np.float64, order="C")
    r = ctx.lm_batch(f, case["row_off"], Xv, None if jac_mode == capi.JAC_ANALYTIC else np.full(n, prm["dx"]), prm["lambda0"],
                     prm["factor"], prm["xmindiff"], prm["maxiter"], jac_mode, want_F=True)
    f.close()
    return r


def check_problem(got, b, want, row_off):
    lo, hi = row_off[b], row_off[b + 1]
    assert _same(got["X"][b], want["X"]), (b, got["X"][b], want["X"])
    assert _same(got["chisq"][b], want["chisq"]) and _same(got["lam"][b], want["lam"]), b
    assert got["iters"][b] == want["iters"] and got["stopped"][b] == want["stopped"], (b, got["iters"][b], want["iters"])
    assert _same(got["F"][lo:hi], want["F"]), b


BUILTINS = [("expcurve", capi.F_EXPCURVE, 3), ("cubic", capi.F_CUBIC, 4)] + \
           [("lorentz%d" % K, capi.F_LORENTZ_SUM, 2 * K) for K in (1, 2, 4, 8, 16)]


@pytest.mark.parametrize("name,kind,n", BUILTINS, ids=[c[0] for c in BUILTINS])
def test_builtin_parity_forward_difference(ctx, name, kind, n):
    """ragged m_b in {0, 1, n - 1, n, 2048, ...}: rank-deficient problems (m_b < n) take NaN steps and reject them all"""
    sizes = [0, 1, n - 1, n, 2048, 37, 300, 5]
    case = LC.make_batch(kind, n, sizes, seed=n + kind)
    got = run(ctx, case)
    for b in range(len(sizes)):
        check_problem(got, b, LC.oracle_problem(case, b, PRM["lambda0"], PRM["factor"], PRM["dx"], PRM["maxiter"], PRM["xmindiff"]),
                      case["row_off"])
    assert got["stopped"].any() and not got["stopped"].all()      # early stops next to problems that run to max_iter


@pytest.mark.parametrize("maxiter,xmindiff", [(0, 1e-9), (25, 0.0)])
def test_max_iter_zero_and_x_min_diff_zero(ctx, maxiter, xmindiff):
    case = LC.make_batch(capi.F_LORENTZ_SUM, 4, [100, 7, 0, 64], seed=2)
    got = run(ctx, case, maxiter=maxiter, xmindiff=xmindiff)
    for b in range(4):
        check_problem(got, b, LC.oracle_problem(case, b, PRM["lambda0"], PRM["factor"], PRM["dx"], maxiter, xmindiff), case["row_off"])
    if maxiter == 0:
        assert _same(got["X"], case["X0"]) and np.all(got["lam"] == PRM["lambda0"]) and np.all(got["iters"] == 0)


def _user():
    import user_jacobian_lib as UJ
    UJ.build_and_load()
    return UJ


def _host_model(UJ, kind, case, b):
    cols, m = LC.problem_columns(case, b)
    resid = lambda x: UJ.host_jacobian(kind, case["scalars"], cols, x)[1]
    jac = lambda x, F: UJ.host_jacobian(kind, case["scalars"], cols, x)[0]
    return resid, jac


@pytest.mark.parametrize("name,kind,n", BUILTINS + [("user_lorentz", 2101, 8), ("user_gauss", 2102, 3)],
                         ids=[c[0] for c in BUILTINS] + ["user_lorentz", "user_gauss"])
def test_analytic_parity(ctx, name, kind, n):
    UJ = _user()
    sizes = [0, 2, n, 500, 41]
    case = LC.make_batch(kind, n, sizes, seed=3 * n + kind)
    got = run(ctx, case, jac_mode=capi.JAC_ANALYTIC)
    for b in range(len(sizes)):
        resid, jac = _host_model(UJ, kind, case, b)
        check_problem(got, b, LC.py_lm(resid, jac, case["X0"][b], PRM["lambda0"], PRM["factor"], PRM["maxiter"], PRM["xmindiff"]),
                      case["row_off"])


def test_user_models_forward_difference(ctx):
    UJ = _user()
    case = LC.make_batch(2101, 8, [0, 3, 700, 64], seed=11)         # the user copy of the sum of Lorentzians: the oracle knows its model
    got = run(ctx, case)
    for b in range(4):
        check_problem(got, b, LC.oracle_problem(case, b, PRM["lambda0"], PRM["factor"], PRM["dx"], PRM["maxiter"], PRM["xmindiff"],
                                                kind=capi.F_LORENTZ_SUM), case["row_off"])
    case = LC.make_batch(2102, 3, [0, 1, 3, 400], seed=12)          # the Gaussian peak: the Python loop over its host residual
    got = run(ctx, case)
    for b in range(4):
        resid, _ = _host_model(UJ, 2102, case, b)
        check_problem(got, b, LC.py_lm(resid, LC.fd_jac(resid, PRM["dx"]), case["X0"][b], PRM["lambda0"], PRM["factor"], PRM["maxiter"],
                                       PRM["xmindiff"]), case["row_off"])
    # a model without jacobian(): the batch launcher refuses the analytic mode
    f = ctx.functor(2104, (0.1,), (), case["columns"], case["columns"][0].size)
    with pytest.raises(capi.PnolError, match="NO_FUNCTOR"):
        ctx.lm_batch(f, case["row_off"], case["X0"].copy(), None, jac_mode=capi.JAC_ANALYTIC)


def lorentz_uniform(B, K, mb, seed):
    """B sum-of-Lorentzians problems of mb rows each, generated at once"""
    rng = np.random.default_rng(seed)
    t1 = np.linspace(-0.5, 1.5, mb)
    a = rng.uniform(1, 2, (B, K))
    c = (np.arange(K) + rng.uniform(0.3, 0.7, (B, K))) / K
    y = np.zeros((B, mb))
    for k in range(K):
        y += a[:, k:k + 1] / (1 + LC.LORENTZ_W * (t1[None, :] - c[:, k:k + 1]) ** 2)
    X0 = np.empty((B, 2 * K))
    X0[:, 0::2] = a * rng.uniform(0.9, 1.1, (B, K))
    X0[:, 1::2] = c + rng.uniform(-0.02, 0.02, (B, K)) / K
    return dict(kind=capi.F_LORENTZ_SUM, n=2 * K, scalars=(LC.LORENTZ_W,), columns=[np.tile(t1, B), y.ravel()],
                row_off=np.arange(B + 1, dtype=np.int64) * mb, X0=X0)


@pytest.mark.parametrize("B,K,mb", [(1 << 20, 2, 32), (65536, 16, 1024)], ids=["1M_n4", "64k_n32"])
def test_scale_random_sample(ctx, B, K, mb):
    case = lorentz_uniform(B, K, mb, seed=B + K)
    got = run(ctx, case, maxiter=8)
    for b in np.random.default_rng(1).choice(B, 256, replace=False):
        check_problem(got, b, LC.oracle_problem(case, b, PRM["lambda0"], PRM["factor"], PRM["dx"], 8, PRM["xmindiff"]), case["row_off"])


def test_independence_of_batch_size_position_and_neighbours(ctx):
    B, K, mb = 65536, 2, 64
    case = lorentz_uniform(B, K, mb, seed=5)
    full = run(ctx, case, maxiter=12)
    perm = np.random.default_rng(2).permutation(B)
    cols = [c.reshape(B, mb)[perm].ravel() for c in case["columns"]]
    pcase = dict(case, columns=cols, X0=case["X0"][perm])
    permuted = run(ctx, pcase, maxiter=12)
    inv = np.argsort(perm)
    for k in ("X", "chisq", "lam", "iters", "stopped"):
        assert np.array_equal(np.asarray(permuted[k])[inv].view(np.uint8), np.asarray(full[k]).view(np.uint8)), k
    for b in (0, 1234, B - 1):
        alone = dict(case, columns=[c[b * mb:(b + 1) * mb].copy() for c in case["columns"]], row_off=np.array([0, mb]), X0=case["X0"][b:b + 1])
        one = run(ctx, alone, maxiter=12)
        assert _same(one["X"][0], full["X"][b]) and _same(one["chisq"][0], full["chisq"][b]) and one["iters"][0] == full["iters"][b]


def test_device_pointers_misaligned_x_and_prefilled_outputs(ctx):
    import torch
    case = LC.make_batch(capi.F_CUBIC, 4, [40, 0, 90, 4], seed=21)
    want = run(ctx, case)
    dev = torch.device("cuda:0")
    dcols = [torch.tensor(c, device=dev) for c in case["columns"]]            # borrowed by the functor: kept alive here
    f = ctx.functor(capi.F_CUBIC, (), (), dcols, case["columns"][0].size)
    store = torch.full((1 + case["X0"].size,), float("nan"), dtype=torch.float64, device=dev)
    Xd = store[1:]                                                  # 8 bytes past the allocation: not 16-byte aligned
    Xd.copy_(torch.tensor(case["X0"].ravel(), device=dev))
    out = dict(chisq=torch.full((4,), float("nan"), dtype=torch.float64, device=dev), lam=torch.full((4,), float("nan"), dtype=torch.float64, device=dev),
               iters=torch.full((4,), -7, dtype=torch.int32, device=dev), stopped=torch.full((4,), -7, dtype=torch.int32, device=dev),
               F=torch.full((case["columns"][0].size,), float("nan"), dtype=torch.float64, device=dev))
    r = ctx.lm_batch(f, torch.tensor(case["row_off"], device=dev), Xd, torch.full((4,), PRM["dx"], dtype=torch.float64, device=dev),
                     PRM["lambda0"], PRM["factor"], PRM["xmindiff"], PRM["maxiter"], n=4, B=4, out=out)
    torch.cuda.synchronize()
    assert _same(Xd.cpu().numpy().reshape(4, 4), want["X"])
    for k in ("chisq", "lam", "F"):
        assert _same(r[k].cpu().numpy(), want[k]), k
    assert np.array_equal(r["iters"].cpu().numpy(), want["iters"]) and np.array_equal(r["stopped"].cpu().numpy(), want["stopped"])
    # host outputs prefilled with NaN: F rows outside every problem keep their NaN
    hf = ctx.functor(capi.F_CUBIC, (), (), case["columns"], case["columns"][0].size)
    ro = case["row_off"].copy()
    ro[0] = 10                                                      # problem 0 starts at row 10: rows 0 .. 9 belong to none
    outs = dict(chisq=np.full(4, np.nan), lam=np.full(4, np.nan), iters=np.full(4, -7, np.int32), stopped=np.full(4, -7, np.int32),
                F=np.full(case["columns"][0].size, np.nan))
    r = ctx.lm_batch(hf, ro, case["X0"].copy(), np.full(4, PRM["dx"]), PRM["lambda0"], PRM["factor"], PRM["xmindiff"], PRM["maxiter"], out=outs)
    assert np.all(np.isnan(r["F"][:10])) and not np.any(np.isnan(r["chisq"])) and np.all(r["iters"] >= 0)
    assert _same(r["X"][1:], want["X"][1:])


def test_refusals(ctx):
    case = LC.make_batch(capi.F_EXPCURVE, 3, [20, 30], seed=4)
    f = ctx.functor(capi.F_EXPCURVE, (), (), case["columns"], 50)
    dx = np.full(3, 1e-7)

    def call(**kw):
        a = dict(row_off=case["row_off"], X=case["X0"].copy(), dx=dx)
        a.update(kw)
        return ctx.lm_batch(f, a["row_off"], a["X"], a["dx"])

    for bad in ([0, 30, 20], [-1, 20, 50], [0, 20, 51]):
        with pytest.raises(capi.PnolError, match="INVALID"):
            call(row_off=np.array(bad))
    with pytest.raises(capi.PnolError, match="INVALID"):
        call(dx=None)
    with pytest.raises(capi.PnolError, match="INVALID"):
        ctx.lm_batch(f, np.arange(3) * 20, np.zeros((2, 65)), np.full(65, 1e-7))
    with pytest.raises(capi.PnolError, match="INVALID"):
        ctx.lm_batch(ctx.functor(capi.F_ROSENBROCK), case["row_off"], case["X0"].copy(), dx)
    lz = ctx.functor(capi.F_LORENTZ_SUM, (40.0,), (), case["columns"][:2], 50)
    with pytest.raises(capi.PnolError, match="INVALID"):
        ctx.lm_batch(lz, case["row_off"], np.ones((2, 6)), np.full(6, 1e-7))     # K = 3 is not a power of two
    r = ctx.lm_batch(f, np.zeros(1, dtype=np.int64), np.zeros((0, 3)), dx)        # B = 0: a no-op
    assert r["X"].shape == (0, 3)


def test_plugin_class_equals_c_abi_and_fits(ctx):
    from parallelnonlinearoptimizationlibrary_b200 import hostapi
    hostapi.attach(ctx)
    try:
        case = LC.make_batch(capi.F_LORENTZ_SUM, 8, [512] * 16 + [3, 0], seed=8)
        for mode in (capi.JAC_AUTO, capi.JAC_ANALYTIC):
            hostapi.set_jac_mode(mode)
            h = hostapi.lm_batch_lorentz(case["columns"][0], case["columns"][1], LC.LORENTZ_W, case["row_off"], case["X0"], dxgrad=PRM["dx"],
                                         maxiter=100, xmindiff=PRM["xmindiff"])
            c = run(ctx, case, jac_mode=mode, maxiter=100)
            for k in ("X", "chisq", "lam", "iters", "stopped"):
                assert np.array_equal(np.asarray(h[k]).view(np.uint8), np.asarray(c[k]).view(np.uint8)), (mode, k)
            assert np.max(np.abs(h["X"][:16] - case["Xtrue"][:16])) < 1e-2, mode
        hostapi.set_jac_mode(capi.JAC_AUTO)
        one = LC.make_batch(capi.F_EXPCURVE, 3, [80], seed=6)
        s = hostapi.lm_batch_single(capi.F_EXPCURVE, (), one["columns"], one["X0"][0], dxgrad=PRM["dx"], maxiter=PRM["maxiter"],
                                    xmindiff=PRM["xmindiff"])
        want = LC.oracle_problem(one, 0, PRM["lambda0"], PRM["factor"], PRM["dx"], PRM["maxiter"], PRM["xmindiff"])
        assert _same(s["X"], want["X"]) and _same(s["F"], want["F"]) and _same(s["F0"], want["F0"])
    finally:
        hostapi.set_jac_mode(capi.JAC_AUTO)
        hostapi.detach()


def test_two_gpus_give_the_one_gpu_bits(ctx):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    B, K, mb = 4096, 4, 128
    case = lorentz_uniform(B, K, mb, seed=17)
    whole = run(ctx, case, maxiter=15)
    h = B // 2
    parts = []
    for dev, sl in ((0, slice(0, h)), (1, slice(h, B))):
        c2 = capi.Context(dev)
        part = dict(case, columns=[c.reshape(B, mb)[sl].ravel() for c in case["columns"]], row_off=np.arange(h + 1, dtype=np.int64) * mb,
                    X0=case["X0"][sl])
        parts.append(run(c2, part, maxiter=15))
        c2.close()
    for k in ("X", "chisq", "lam", "iters", "stopped", "F"):
        assert np.array_equal(np.concatenate([np.asarray(p[k]) for p in parts]).view(np.uint8), np.asarray(whole[k]).view(np.uint8)), k
