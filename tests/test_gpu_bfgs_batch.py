"""Batched BFGS on the GPU (pnol_bfgs_batch): every field of every start bit for bit the CPU stand-in's oracle_bfgs
(tests/host_logic_bfgs_batch.cpp), which tests/test_bfgs_batch_cpu.py pins bit for bit to the unmodified host BFGS controller, for the
six built-in objectives, all eight derivative-flag combinations and both initial inverse Hessians; the user kinds; independence from
B, position and order; random samples at 65 536 and 2^20 starts; host, device and misaligned pointers; the refusals; the plugin class;
and a batch split over two GPUs."""
import numpy as np
import pytest

import bfgs_batch_cases as BC
import host_logic_bfgs_batch_lib as HLB
from parallelnonlinearoptimizationlibrary_b200 import capi, hostapi

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    hostapi.attach(c)
    yield c
    hostapi.detach()
    c.close()


@pytest.fixture(scope="module")
def standin():
    hl = HLB.build_and_load()
    if hl is None:
        pytest.skip("no g++ on this box")
    return hl


def check_same(got, want, where):
    for key in ("X", "f0", "fopt"):
        assert BC.same(got[key], want[key]), (where, key, BC.diff_report(got[key], want[key]))
    assert np.array_equal(got["iters"], want["iters"]) and np.array_equal(got["stop"], want["stop"]), where


STOPS_SEEN = set()


@pytest.mark.parametrize("flags", BC.FLAG_SETS)
@pytest.mark.parametrize("name", sorted(BC.OBJECTIVES))
def test_builtin_parity(ctx, standin, name, flags):
    """the plugin class on the GPU against the same class on the stand-in, for every dimension of the objective"""
    for n in BC.OBJECTIVES[name][2]:
        for ih in (0, 1):
            prm = BC.params(init_hess_fd=ih)
            X = BC.starts(name, n, 48, seed=n + 31 * ih + flags)
            st, got = BC.run_batch(hostapi.lib(), name, X, prm, flags)
            assert st == 0, hostapi.lib().pnolhost_last_error()
            st, want = BC.run_batch(standin, name, X, prm, flags)
            assert st == 0
            check_same(got, want, (name, n, flags, ih))
            STOPS_SEEN.update(int(s) for s in got["stop"])


def test_every_stop_code_occurs():
    """the grid above ends starts by max_iter (0), by xdiff (1) and by the gradient norm (2)"""
    if not STOPS_SEEN:
        pytest.skip("runs after test_builtin_parity")
    assert STOPS_SEEN == {0, 1, 2}


@pytest.mark.parametrize("edge", [dict(max_iter=0), dict(max_iter_ls=0), dict(max_iter_ls=1), dict(x_min_diff=0.0, min_grad_2norm=0.0)])
def test_edge_parameters(ctx, standin, edge):
    for name, n in (("rosenbrock", 8), ("rastrigin", 16), ("goldstein", 2)):
        for flags in (0, 7):
            prm = BC.params(init_hess_fd=1, **edge)
            X = BC.starts(name, n, 16, seed=5)
            got = BC.run_batch(hostapi.lib(), name, X, prm, flags)[1]
            want = BC.run_batch(standin, name, X, prm, flags)[1]
            check_same(got, want, (name, edge, flags))


def _c_abi(ctx, kind, X, flags=0, ints=(), **kw):
    f = ctx.functor(kind, (), ints)
    prm = dict(BC.PRM, **kw)
    prm["init_hess_fd"] = bool(prm["init_hess_fd"])
    return ctx.bfgs_batch(f, np.array(X, dtype=np.float64), flags=flags, **prm)


def test_c_abi_equals_the_plugin_class(ctx, standin):
    X = BC.starts("rosenbrock", 8, 40, seed=9)
    for flags in (0, 3, 7):
        got = _c_abi(ctx, capi.F_ROSENBROCK, X, flags, init_hess_fd=1)
        want = BC.run_batch(standin, "rosenbrock", X, BC.params(init_hess_fd=1), flags)[1]
        check_same(dict(got, fopt=got["fopt"]), want, flags)


def test_independence_of_batch_size_position_and_order(ctx):
    X = BC.starts("rastrigin", 16, 300, seed=4)
    whole = _c_abi(ctx, capi.F_RASTRIGIN, X, 3)
    perm = np.random.default_rng(1).permutation(300)
    shuffled = _c_abi(ctx, capi.F_RASTRIGIN, X[perm], 3)
    for key in ("X", "f0", "fopt", "iters", "stop"):
        assert BC.same(np.asarray(shuffled[key], dtype=np.float64), np.asarray(whole[key], dtype=np.float64)[perm]), key
    for b in (0, 123, 299):
        one = _c_abi(ctx, capi.F_RASTRIGIN, X[b:b + 1], 3)
        assert BC.same(one["X"][0], whole["X"][b]) and BC.same(one["fopt"][0], whole["fopt"][b]) and one["iters"][0] == whole["iters"][b]
    big = _c_abi(ctx, capi.F_RASTRIGIN, np.concatenate([X[:1]] * 5000), 3)
    assert np.all(big["X"].view(np.uint64) == whole["X"][0].view(np.uint64)) and np.all(big["iters"] == whole["iters"][0])


@pytest.mark.parametrize("B", [65536, 1 << 20])
def test_scale_random_sample(ctx, standin, B):
    import torch
    n = 16
    rng = np.random.default_rng(B)
    X = rng.uniform(-5.12, 5.12, size=(B, n))
    Xd = torch.tensor(X, device="cuda:0")
    f = ctx.functor(capi.F_RASTRIGIN)
    out = dict(f0=torch.empty(B, dtype=torch.float64, device="cuda:0"), fopt=torch.empty(B, dtype=torch.float64, device="cuda:0"),
               iters=torch.empty(B, dtype=torch.int32, device="cuda:0"), stop=torch.empty(B, dtype=torch.int32, device="cuda:0"))
    prm = dict(BC.PRM)
    prm["init_hess_fd"] = False
    ctx.bfgs_batch(f, Xd, flags=3, n=n, B=B, out=out, **prm)
    got = dict(X=Xd.cpu().numpy(), **{k: v.cpu().numpy() for k, v in out.items()})
    idx = np.sort(rng.choice(B, size=256 if B == 65536 else 64, replace=False))
    want = BC.run_batch(standin, "rastrigin", X[idx], BC.params(), 3)[1]
    check_same({k: v[idx] for k, v in got.items()}, want, B)


def test_host_device_and_misaligned_pointers(ctx):
    import torch
    X = BC.starts("goldstein", 2, 64, seed=8)
    want = _c_abi(ctx, capi.F_GOLDSTEIN, X, 7, init_hess_fd=1)
    f = ctx.functor(capi.F_GOLDSTEIN)
    store = torch.full((1 + X.size,), float("nan"), dtype=torch.float64, device="cuda:0")
    Xd = store[1:]                                                  # 8 bytes past the allocation: not 16-byte aligned
    Xd.copy_(torch.tensor(X.ravel(), device="cuda:0"))
    ostore = torch.full((1 + 2 * 64,), float("nan"), dtype=torch.float64, device="cuda:0")
    istore = torch.full((1 + 2 * 64,), -7, dtype=torch.int32, device="cuda:0")
    out = dict(f0=ostore[1:65], fopt=ostore[65:], iters=istore[1:65], stop=istore[65:])
    prm = dict(BC.PRM, init_hess_fd=True)
    ctx.bfgs_batch(f, Xd, flags=7, n=2, B=64, out=out, **prm)
    assert BC.same(Xd.cpu().numpy().reshape(64, 2), want["X"])
    for k in ("f0", "fopt", "iters", "stop"):
        assert BC.same(out[k].cpu().numpy().astype(np.float64), np.asarray(want[k], dtype=np.float64)), k


def test_refusals(ctx):
    f = ctx.functor(capi.F_ROSENBROCK)
    X = np.zeros((4, 3))

    def status(fn):
        try:
            fn()
            return capi.PNOL_OK, ""
        except capi.PnolError as e:
            return e.args[0].split(":")[0], str(e)

    assert status(lambda: ctx.bfgs_batch(f, X, n=0, B=4))[0] == "INVALID"
    st, msg = status(lambda: ctx.bfgs_batch(f, np.zeros((4, 65))))
    assert st == "INVALID" and "outside 1 .. 64" in msg
    assert status(lambda: ctx.bfgs_batch(f, X, n=3, B=-1))[0] == "INVALID"
    st, msg = status(lambda: ctx.bfgs_batch(f, X, prm="null"))
    assert st == "INVALID" and "prm" in msg
    st, msg = status(lambda: ctx.bfgs_batch(f, 0, n=3, B=4))
    assert st == "INVALID" and "required" in msg
    assert status(lambda: ctx.bfgs_batch(f, np.zeros((0, 3)), n=3, B=0))[0] == capi.PNOL_OK     # B = 0: a no-op
    t = np.linspace(0, 1, 10)
    r = ctx.functor(capi.F_EXPCURVE, (), (), (t, t), 10)
    st, msg = status(lambda: ctx.bfgs_batch(r, X))
    assert st == "NO_FUNCTOR" and "not a scalar objective" in msg


def test_user_kinds(ctx):
    import user_functor_lib as U
    import user_gradient_lib as UG
    import user_hessian_lib as UH
    U.build_and_load(); UG.build_and_load(); UH.build_and_load()
    n = 6
    rng = np.random.default_rng(2)
    X = rng.uniform(-3, 3, size=(32, n))
    trid_min = np.array([i * (n + 1 - i) for i in range(1, n + 1)], dtype=np.float64)
    ft = ctx.functor(UG.MYG_F_TRID)
    for flags in (0, 1, 3):
        got = ctx.bfgs_batch(ft, X.copy(), flags=flags, max_iter=200, x_min_diff=1e-12, min_grad_2norm=1e-8)
        assert np.max(np.abs(got["X"] - trid_min)) < 1e-3, flags
    fs = ctx.functor(UG.MYG_F_STYBLINSKI, (0.5,))
    for flags in (0, 3):
        got = ctx.bfgs_batch(fs, X.copy(), flags=flags, max_iter=200, x_min_diff=1e-12, min_grad_2norm=1e-8)
        # every coordinate at one of the two stationary points of a well, -2.9035 or 2.7468
        assert np.all(np.minimum(np.abs(got["X"] + 2.9035), np.abs(got["X"] - 2.7468)) < 1e-3), flags
    M = rng.normal(size=(n, n))
    A = M @ M.T + n * np.eye(n)
    fq = ctx.functor(UH.MYH_F_QUADFORM, (), (), (A.ravel(),), n * n)
    got = ctx.bfgs_batch(fq, X.copy(), flags=4, init_hess_fd=True, max_iter=50)
    # the gradient is the forward difference (the kind has no partial()): its O(dx_grad) bias moves the minimiser by about 1e-6
    assert np.max(np.abs(got["X"])) < 1e-5
    # a kind without partial(): the analytic gradient / slope flags refused, the forward difference accepted
    fn_ = ctx.functor(U.MY_F_TRID)
    for flags in (1, 2):
        with pytest.raises(capi.PnolError, match="NO_FUNCTOR"):
            ctx.bfgs_batch(fn_, X.copy(), flags=flags)
    got = ctx.bfgs_batch(fn_, X.copy(), flags=0, max_iter=200, x_min_diff=1e-12, min_grad_2norm=1e-8)
    assert np.max(np.abs(got["X"] - trid_min)) < 1e-3


def test_plugin_class_single_start(ctx, standin):
    x0 = np.array([-1.2, 1.0, 0.7, 0.2])
    prm = BC.vec(BC.params(max_iter=200))
    got = hostapi.bfgs_batch("rosenbrock", x0, prm, single=True)
    st, want = BC.run_serial(standin, "rosenbrock", x0, BC.params(max_iter=200), 0)
    assert st == 0 and BC.same(got["X"][0], want["X"]) and BC.same(got["fOpt"][0], want["fopt"])
    # and the GPU BFGS class reaches the same minimum (RANK2 / tensor-core products: close, not bit-equal)
    cls = hostapi.bfgs("bfgs", "rosenbrock", x0, prm)
    assert np.max(np.abs(cls["X"] - got["X"][0])) < 1e-3


def test_two_gpus_give_the_one_gpu_bits(ctx):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    X = BC.starts("rosenbrock", 8, 2000, seed=12)
    whole = _c_abi(ctx, capi.F_ROSENBROCK, X, 3)
    c1 = capi.Context(1)
    try:
        f1 = c1.functor(capi.F_ROSENBROCK)
        prm = dict(BC.PRM, init_hess_fd=False)
        part = c1.bfgs_batch(f1, X[1000:].copy(), flags=3, **prm)
    finally:
        c1.close()
    first = _c_abi(ctx, capi.F_ROSENBROCK, X[:1000], 3)
    assert BC.same(np.concatenate([first["X"], part["X"]]), whole["X"])
    assert np.array_equal(np.concatenate([first["iters"], part["iters"]]), whole["iters"])
