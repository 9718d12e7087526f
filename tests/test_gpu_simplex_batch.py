"""Batched simplex search on the GPU (pnol_simplex_batch): every field of every start bit for bit the CPU stand-in's oracle_simplex
(tests/host_logic_standin.cpp), which tests/test_simplex_batch_cpu.py pins bit for bit to the unmodified host SimplexSearch
controller, for the six built-in objectives with counter and explicit streams and for user objectives that drive simplexSort into its
quirks; the plugin class on the verbatim reference's golden cases; independence from B, position and stream offset; random samples at
65 536 and 2^20 starts; host, device and misaligned pointers; the refusals; and a batch split over two GPUs."""
import os
import sys

import numpy as np
import pytest

import host_standin
import simplex_batch_cases as SC
from parallelnonlinearoptimizationlibrary_b200 import capi, hostapi

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def ctx():
    c = capi.Context(0)
    hostapi.attach(c)
    yield c
    hostapi.detach()
    c.close()


@pytest.fixture(scope="module")
def standin():
    hl = host_standin.load()
    if hl is None:
        pytest.skip("no g++ on this box")
    return hl


def check_same(got, want, where):
    for key in ("X", "f0", "fopt"):
        assert SC.same(got[key], want[key]), (where, key, SC.diff_report(got[key], want[key]))
    for key in ("iters", "stop", "evals"):
        assert np.array_equal(np.asarray(got[key]), np.asarray(want[key])), (where, key)


def gpu(ctx, kind, X, prm, stream, offset=0, ints=(), scalars=()):
    f = ctx.functor(kind, tuple(scalars), tuple(ints))
    if stream[0] == "values":
        s = stream[1]
    elif stream[0] == "device":
        s = stream[1]
    else:
        s = capi.StreamDesc(None, 0, int(stream[1]), float(stream[2]))
    return ctx.simplex_batch(f, np.array(X, dtype=np.float64), stream=s, stream_offset=offset, **prm)


STOPS_SEEN = set()


@pytest.mark.parametrize("stream_kind", ["seed", "values", "device"])
@pytest.mark.parametrize("name", sorted(SC.OBJECTIVES))
def test_builtin_parity(ctx, standin, name, stream_kind):
    import torch
    kind, ints = SC.kind_of(name)
    for n in SC.OBJECTIVES[name][2]:
        B = 48
        X = SC.starts(name, n, B, seed=n + 5)
        prm = SC.params(max_iter=400 if n <= 16 else 150)
        if stream_kind == "seed":
            stream = ("seed", 31 + n, 1.0)
            gs = stream
        else:
            vals = np.random.default_rng(n).uniform(size=B * n * n)
            stream = ("values", vals)
            gs = ("values", vals) if stream_kind == "values" else ("device", torch.tensor(vals, device="cuda:0"))
        if name == "expsingle":
            # its data columns come with the example objective: the plugin class on both sides (explicit streams from the host)
            st, got = SC.run_batch(hostapi.lib(), name, X, prm, stream)
            assert st == 0, hostapi.lib().pnolhost_last_error()
            hostapi.clear_stream()
            st, want = SC.run_batch(standin, name, X, prm, stream)
        else:
            got = gpu(ctx, kind, X, prm, gs, ints=ints)
            st, want = SC.run_standin_capi(standin, kind, X, prm, stream, ints=ints)
        assert st == 0
        check_same(got, want, (name, n, stream_kind))
        STOPS_SEEN.update(int(s) for s in got["stop"])


def test_both_stop_codes_occur():
    if not STOPS_SEEN:
        pytest.skip("runs after test_builtin_parity")
    assert STOPS_SEEN == {0, 1}


@pytest.mark.parametrize("kw", [dict(alpha=1.3, gamma=2.7, rho=0.35, sigma=0.8), dict(max_iter=0), dict(max_iter=1),
                                dict(x_min_diff=0.0, max_iter=200), dict(init_rand_max=0.0), dict(init_rand_max=4.0, sigma=0.9)])
def test_parameters(ctx, standin, kw):
    for name, n in (("rosenbrock", 8), ("rastrigin", 16), ("goldstein", 2), ("rosenbrock", 64)):
        kind, ints = SC.kind_of(name)
        X = SC.starts(name, n, 24, seed=7)
        prm = SC.params(**kw)
        stream = ("seed", 5, 1.0)
        got = gpu(ctx, kind, X, prm, stream, ints=ints)
        want = SC.run_standin_capi(standin, kind, X, prm, stream, ints=ints)[1]
        check_same(got, want, (name, n, kw))


def test_user_kinds_take_the_quirk_paths(ctx, standin):
    import user_simplex_lib as US
    US.build_and_load()
    rng = np.random.default_rng(3)
    for kind, name in sorted(US.NAMES.items()):
        irregular = 0
        for n in (1, 2, 5, 16, 40):
            X = rng.uniform(-1.5, 2.5, size=(64, n))
            prm = SC.params(max_iter=300, init_rand_max=1.5)
            for stream in (("seed", kind + n, 1.0), ("values", rng.uniform(size=64 * n * n))):
                before = standin.standin_simplex_irregular_sorts()
                st, want = SC.run_standin_capi(standin, kind, X, prm, stream)
                assert st == 0
                irregular += standin.standin_simplex_irregular_sorts() - before
                got = gpu(ctx, kind, X, prm, stream)
                check_same(got, want, (name, n, stream[0]))
        # the oracle's count: these objectives took simplexSort outside its regime (sentinels, repeated vertices)
        if name in ("negative", "signed_zero", "nan_region"):
            assert irregular > 0, name


def test_plugin_class_single_start_is_the_verbatim_reference(ctx):
    """SimplexSearchBatch's base-class findMin (B = 1) on every case of tests/golden/simplex_golden.npz returns the verbatim
    reference's bits"""
    sys.path.insert(0, os.path.join(HERE, "golden"))
    from make_simplex_golden import CASES
    G = np.load(os.path.join(HERE, "golden", "simplex_golden.npz"))
    try:
        for name, (obj, x0, kw, stream) in CASES.items():
            if stream[0] == "values":
                hostapi.set_stream(values=stream[1])
            else:
                hostapi.set_stream(seed=stream[1], scale=stream[2])
            r = hostapi.simplex_batch(obj, x0, alpha=kw.get("alpha", 1.0), gamma=kw.get("gamma", 2.0), rho=kw.get("rho", 0.5),
                                      sigma=kw.get("sigma", 0.5), maxiter=kw.get("maxiter", 10000), init_rand_max=kw.get("initrandmax", 1.0),
                                      xmindiff=kw.get("xmindiff", 1e-7), single=True)
            assert np.array_equal(r["X"][0], G[name + "/X"]), name
            assert r["f0"][0] == G[name + "/f0"][0] and r["fOpt"][0] == G[name + "/fOpt"][0], name
            assert r["stream_pos"] == int(G[name + "/stream_pos"][0]), name
            # and the reports of findMin(X, reports) on the same start
            full = hostapi.simplex_batch(obj, x0, alpha=kw.get("alpha", 1.0), gamma=kw.get("gamma", 2.0), rho=kw.get("rho", 0.5),
                                         sigma=kw.get("sigma", 0.5), maxiter=kw.get("maxiter", 10000), init_rand_max=kw.get("initrandmax", 1.0),
                                         xmindiff=kw.get("xmindiff", 1e-7))
            assert np.array_equal(full["X"][0], G[name + "/X"]) and full["fOpt"][0] == G[name + "/fOpt"][0], name
    finally:
        hostapi.clear_stream()


def test_independence_of_batch_size_position_and_offset(ctx, standin):
    X = SC.starts("rastrigin", 16, 300, seed=4)
    prm = SC.params(max_iter=300)
    stream = ("seed", 17, 1.0)
    whole = gpu(ctx, capi.F_RASTRIGIN, X, prm, stream)
    parts = [gpu(ctx, capi.F_RASTRIGIN, X[a:b], prm, stream, offset=a * 256) for a, b in ((0, 1), (1, 77), (77, 300))]
    for key in ("X", "f0", "fopt", "iters", "stop", "evals"):
        cat = np.concatenate([np.asarray(p[key], dtype=np.float64) for p in parts])
        assert SC.same(cat, np.asarray(whole[key], dtype=np.float64)), key
    for b in (0, 123, 299):
        one = gpu(ctx, capi.F_RASTRIGIN, X[b:b + 1], prm, stream, offset=b * 256)
        assert SC.same(one["X"][0], whole["X"][b]) and SC.same(one["fopt"][0], whole["fopt"][b]) and one["iters"][0] == whole["iters"][b]
    # one explicit stream holding start 0's draws 5000 times over: every start equals start 0
    vals = np.tile(SC.draws(standin, stream, 0, 256), 5000)
    big = gpu(ctx, capi.F_RASTRIGIN, np.concatenate([X[:1]] * 5000), prm, ("values", vals))
    assert np.all(big["X"].view(np.uint64) == whole["X"][0].view(np.uint64)) and np.all(big["iters"] == whole["iters"][0])


@pytest.mark.parametrize("B", [65536, 1 << 20])
def test_scale_random_sample(ctx, standin, B):
    import torch
    n = 8
    rng = np.random.default_rng(B)
    X = rng.uniform(-2.0, 2.0, size=(B, n))
    Xd = torch.tensor(X, device="cuda:0")
    f = ctx.functor(capi.F_ROSENBROCK)
    out = dict(f0=torch.empty(B, dtype=torch.float64, device="cuda:0"), fopt=torch.empty(B, dtype=torch.float64, device="cuda:0"),
               iters=torch.empty(B, dtype=torch.int32, device="cuda:0"), stop=torch.empty(B, dtype=torch.int32, device="cuda:0"),
               evals=torch.empty(B, dtype=torch.int64, device="cuda:0"))
    prm = SC.params(max_iter=500)
    ctx.simplex_batch(f, Xd, stream=capi.StreamDesc(None, 0, 99, 1.0), n=n, B=B, out=out, **prm)
    got = dict(X=Xd.cpu().numpy(), **{k: v.cpu().numpy() for k, v in out.items()})
    idx = np.sort(rng.choice(B, size=256 if B == 65536 else 64, replace=False))
    for b in idx:
        want = SC.run_standin_capi(standin, capi.F_ROSENBROCK, X[b:b + 1], prm, ("seed", 99, 1.0), offset=int(b) * n * n)[1]
        check_same({k: v[b:b + 1] for k, v in got.items()}, want, (B, int(b)))


def test_host_device_and_misaligned_pointers(ctx):
    import torch
    X = SC.starts("goldstein", 2, 64, seed=8)
    prm = SC.params()
    vals = np.random.default_rng(8).uniform(size=64 * 4 + 1)
    want = gpu(ctx, capi.F_GOLDSTEIN, X, prm, ("values", vals[1:]))
    f = ctx.functor(capi.F_GOLDSTEIN)
    store = torch.full((1 + X.size,), float("nan"), dtype=torch.float64, device="cuda:0")
    Xd = store[1:]                                                  # 8 bytes past the allocation: not 16-byte aligned
    Xd.copy_(torch.tensor(X.ravel(), device="cuda:0"))
    vd = torch.tensor(vals, device="cuda:0")[1:]                    # a misaligned explicit stream on the device
    ostore = torch.full((1 + 2 * 64,), float("nan"), dtype=torch.float64, device="cuda:0")
    istore = torch.full((1 + 2 * 64,), -7, dtype=torch.int32, device="cuda:0")
    estore = torch.full((1 + 64,), -7, dtype=torch.int64, device="cuda:0")
    out = dict(f0=ostore[1:65], fopt=ostore[65:], iters=istore[1:65], stop=istore[65:], evals=estore[1:])
    ctx.simplex_batch(f, Xd, stream=vd, n=2, B=64, out=out, **prm)
    assert SC.same(Xd.cpu().numpy().reshape(64, 2), want["X"])
    for k in ("f0", "fopt", "iters", "stop", "evals"):
        assert SC.same(out[k].cpu().numpy().astype(np.float64), np.asarray(want[k], dtype=np.float64)), k
    # host X with a misaligned host stream; evals not asked for
    hv = np.empty(vals.size + 1)[1:]
    hv[:] = vals
    got = ctx.simplex_batch(f, X.copy(), stream=hv[1:], want_evals=False, **prm)
    assert SC.same(got["X"], want["X"]) and got["evals"] is None


def test_refusals(ctx):
    f = ctx.functor(capi.F_ROSENBROCK)
    X = np.zeros((4, 3))

    def status(fn):
        try:
            fn()
            return capi.PNOL_OK, ""
        except capi.PnolError as e:
            return e.args[0].split(":")[0], str(e)

    assert status(lambda: ctx.simplex_batch(f, X, n=0, B=4))[0] == "INVALID"
    st, msg = status(lambda: ctx.simplex_batch(f, np.zeros((4, 65))))
    assert st == "INVALID" and "outside 1 .. 64" in msg
    assert status(lambda: ctx.simplex_batch(f, X, n=3, B=-1))[0] == "INVALID"
    st, msg = status(lambda: ctx.simplex_batch(f, X, prm="null"))
    assert st == "INVALID" and "prm" in msg
    st, msg = status(lambda: ctx.simplex_batch(f, X, stream="null"))
    assert st == "INVALID" and "stream" in msg
    st, msg = status(lambda: ctx.simplex_batch(f, 0, n=3, B=4))
    assert st == "INVALID" and "required" in msg
    assert status(lambda: ctx.simplex_batch(f, np.zeros((0, 3)), n=3, B=0))[0] == capi.PNOL_OK     # B = 0: a no-op
    # a stream shorter than stream_offset + B n^2: refused before anything runs, X and the outputs untouched
    Xs = np.full((4, 3), 0.25)
    out = dict(f0=np.full(4, -1.0), fopt=np.full(4, -1.0), iters=np.full(4, -1, dtype=np.int32), stop=np.full(4, -1, dtype=np.int32),
               evals=np.full(4, -1, dtype=np.int64))
    for size, offset in ((35, 0), (36, 1), (10, 11)):
        st, msg = status(lambda: ctx.simplex_batch(f, Xs, stream=np.full(size, 0.5), stream_offset=offset, out=out))
        assert st == "STREAM" and "explicit random stream" in msg
        assert np.all(Xs == 0.25) and all(np.all(v == -1) for v in out.values())
    t = np.linspace(0, 1, 10)
    r = ctx.functor(capi.F_EXPCURVE, (), (), (t, t), 10)
    st, msg = status(lambda: ctx.simplex_batch(r, X))
    assert st == "NO_FUNCTOR" and "not a scalar objective" in msg


def test_two_gpus_give_the_one_gpu_bits(ctx):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    X = SC.starts("rosenbrock", 8, 2000, seed=12)
    prm = SC.params()
    stream = ("seed", 3, 1.0)
    whole = gpu(ctx, capi.F_ROSENBROCK, X, prm, stream)
    c1 = capi.Context(1)
    try:
        f1 = c1.functor(capi.F_ROSENBROCK)
        part = c1.simplex_batch(f1, X[1000:].copy(), stream=capi.StreamDesc(None, 0, 3, 1.0), stream_offset=1000 * 64, **prm)
    finally:
        c1.close()
    first = gpu(ctx, capi.F_ROSENBROCK, X[:1000], prm, stream)
    assert SC.same(np.concatenate([first["X"], part["X"]]), whole["X"])
    assert np.array_equal(np.concatenate([first["iters"], part["iters"]]), whole["iters"])
