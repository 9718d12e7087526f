"""GPU: analytic gradients (pnol_gradient[_recur]) against the host definition of every partial (include/pnol/functors.hpp, the
user's tests/user_functor/my_gradients.hpp) bit for bit; the refusals; the plugin classes with Runtime::setAnalyticGradient(true),
against the same controllers run on the CPU stand-in of tests/test_host_logic_cpu.py extended by the host partials
(tests/host_logic_gradient.cpp); and the column split over 2+ GPUs."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

import host_logic_gradient_lib as HLG
import user_functor_lib as UF
import user_gradient_lib as UG
from parallelnonlinearoptimizationlibrary_b200 import capi

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _nmax():
    import torch
    return int(torch.cuda.get_device_properties(0).shared_memory_per_block_optin) // 8


def _t_y():
    t = np.linspace(-2.0, 3.0, 257)
    return t, 1.5 * np.exp(0.7 * t) + 0.2 + 0.01 * np.sin(7 * t)


# kind, scalars, ints, columns, smallest n, start-point scale
CASES = {
    "rosenbrock": (capi.F_ROSENBROCK, (), (), (), 1, 2.0),
    "power3": (capi.F_POWER, (), (3,), (), 1, 2.0),
    "booth": (capi.F_BOOTH, (), (), (), 2, 3.0),
    "goldstein": (capi.F_GOLDSTEIN, (), (), (), 2, 2.0),
    "rastrigin": (capi.F_RASTRIGIN, (), (), (), 1, 5.12),
    "expsingle": (capi.F_EXPCURVE_SINGLE, (), (), _t_y(), 3, 1.0),
    "user_trid": (UG.MYG_F_TRID, (), (), (), 1, 3.0),
    "user_styblinski": (UG.MYG_F_STYBLINSKI, (0.5,), (), (), 1, 4.0),
}
NS = [1, 2, 3, 31, 32, 33, 1000, 4096, "max"]


@pytest.fixture(scope="module")
def user():
    return UG.build_and_load()


def _functor(ctx, name):
    kind, sc, ints, cols, _, _ = CASES[name]
    return ctx.functor(kind, sc, ints, cols, cols[0].size if cols else 0)


def _host(name, x, idx=None):
    kind, sc, ints, cols, _, _ = CASES[name]
    return UG.host_partials(kind, x, sc, ints, cols, idx)


@pytest.mark.parametrize("name", sorted(CASES))
def test_gradient_is_the_host_partial_bit_for_bit(ctx, user, name):
    import torch
    f = _functor(ctx, name)
    nmin, scale = CASES[name][4], CASES[name][5]
    rng = np.random.default_rng(len(name))
    for n in NS:
        n = _nmax() if n == "max" else n
        if n < nmin:
            continue
        x = rng.uniform(-scale, scale, n)
        want = _host(name, x)
        g, f0 = ctx.gradient(f, x, want_f0=True)
        assert np.array_equal(g, want), (name, n)
        assert f0 == ctx.eval_batch(f, x, 1, n)[0], (name, n)
        g2, none = ctx.gradient(f, x)
        assert np.array_equal(g2, want) and none is None
        if n in (33, 4096) or n == _nmax():
            # device pointers, x misaligned by one double, g prefilled with NaN (every entry is written)
            xb = torch.empty(n + 1, dtype=torch.float64, device="cuda")
            xb[1:] = torch.from_numpy(x).cuda()
            gd = torch.full((n,), float("nan"), dtype=torch.float64, device="cuda")
            torch.cuda.synchronize()
            _, f0d = ctx.gradient(f, xb.data_ptr() + 8, want_f0=True, g=gd.data_ptr(), n=n)
            assert np.array_equal(gd.cpu().numpy(), want) and f0d == f0, (name, n)
    # one coordinate more than fits in shared memory is refused, as by the forward difference
    n = _nmax() + 1
    x = np.full(n, 0.5)
    st = ctx.lib.pnol_gradient(ctx.h, f.handle, capi._ptr(x), n, capi._ptr(np.empty(n)), None)
    st_fd = ctx.lib.pnol_fd_gradient(ctx.h, f.handle, capi._ptr(x), capi._ptr(np.full(n, 1e-7)), n, capi._ptr(np.empty(n)), None)
    assert st == st_fd == capi.ERR_INVALID and b"does not fit" in ctx.lib.pnol_last_error(ctx.h)
    f.close()


@pytest.mark.parametrize("name", ["rosenbrock", "goldstein", "rastrigin", "user_trid", "user_styblinski"])
def test_gradient_recur_is_the_host_partial_at_the_free_coordinates(ctx, user, name):
    f = _functor(ctx, name)
    rng = np.random.default_rng(5)
    for nfull in (2, 40, 1000):
        if nfull < CASES[name][4]:
            continue
        ind = (rng.random(nfull) < 0.3).astype(np.uint8)
        ind[0] = 0
        const_x = rng.uniform(-1, 1, nfull)
        nfree = int((ind == 0).sum())
        for nr in sorted({1, nfree, min(nfull, nfree + 3)}):        # the last: more reduced entries than free variables
            xr = rng.uniform(-1, 1, nr)
            xfull, pos, k = const_x.copy(), np.full(nr, -1, dtype=np.int32), 0
            for j in range(nfull):
                if not ind[j]:
                    xfull[j] = xr[k] if k < nr else 0.0
                    if k < nr:
                        pos[k] = j
                    k += 1
            want = np.zeros(nr)
            has = pos >= 0
            want[has] = _host(name, xfull, pos[has])
            g, f0 = ctx.gradient_recur(f, xr, const_x, ind, want_f0=True)
            assert np.array_equal(g, want), (name, nfull, nr)
            assert f0 == ctx.eval_recur(f, xr, const_x, ind)
            if nr > nfree:
                assert np.all(g[nfree:] == 0.0)
    f.close()


def test_functors_without_a_derivative_are_refused(ctx, user):
    lib = ctx.lib
    UF.build_and_load()
    x, g = np.full(4, 0.5), np.empty(4)
    # a user scalar objective without partial(): refused, never a forward difference; the error names the kind
    ft = ctx.functor(UF.MY_F_TRID)
    assert lib.pnol_gradient(ctx.h, ft.handle, capi._ptr(x), 4, capi._ptr(g), None) == capi.ERR_NO_FUNCTOR
    assert str(UF.MY_F_TRID).encode() in lib.pnol_last_error(ctx.h)
    assert lib.pnol_gradient_recur(ctx.h, ft.handle, capi._ptr(x), 2, capi._ptr(x), capi._ptr(np.array([1, 0, 1, 0], np.uint8)), 4,
                                   capi._ptr(g), None) == capi.ERR_NO_FUNCTOR
    # residual models: refused as the forward difference refuses them
    t, y = _t_y()
    for fr in (ctx.functor(capi.F_EXPCURVE, (), (), (t, y), t.size), ctx.functor(UF.MY_F_GAUSSFIT, (0.3,), (), (t, y), t.size)):
        st = lib.pnol_gradient(ctx.h, fr.handle, capi._ptr(x[:3]), 3, capi._ptr(g), None)
        st_fd = lib.pnol_fd_gradient(ctx.h, fr.handle, capi._ptr(x[:3]), capi._ptr(np.full(3, 1e-7)), 3, capi._ptr(g), None)
        assert st == st_fd != capi.PNOL_OK
    # bad arguments
    fr = ctx.functor(capi.F_ROSENBROCK)
    assert lib.pnol_gradient(ctx.h, fr.handle, capi._ptr(x), 0, capi._ptr(g), None) == capi.ERR_INVALID
    assert lib.pnol_gradient(ctx.h, fr.handle, None, 4, capi._ptr(g), None) == capi.ERR_INVALID


# ---- the plugin classes ----
@pytest.fixture
def host(ctx):
    from parallelnonlinearoptimizationlibrary_b200 import hostapi
    hostapi.attach(ctx)
    hostapi.set_analytic_gradient(True)
    yield hostapi
    hostapi.set_analytic_gradient(False)
    hostapi.set_hinv_mode(capi.HINV_RANK2)
    hostapi.detach()


@pytest.mark.parametrize("obj,name,n", [("rosenbrock", "rosenbrock", 40), ("booth", "booth", 2), ("goldstein", "goldstein", 2),
                                        ("power:3", "power3", 5), ("rastrigin", "rastrigin", 12)])
def test_objective_members_return_the_pnol_gradient_bits(ctx, host, obj, name, n):
    x = np.random.default_rng(n).uniform(-1.5, 1.5, n)
    f = _functor(ctx, name)
    want, _ = ctx.gradient(f, x)
    dx = np.full(n, 1e-7)
    assert np.array_equal(host.gradient(obj, x, dx), want) and np.array_equal(host.gradient(obj, x, dx, mpi=True), want)
    ind = np.zeros(n, np.uint8)
    ind[::3] = 1
    xr = x[ind == 0]
    gr, _ = host.gradient_recur(obj, xr, np.full(xr.size, 1e-7), x, ind)
    assert np.array_equal(gr, ctx.gradient_recur(f, xr, x, ind)[0])
    f.close()


BF = [1e-4, 0.9, 1e-6, 1.0, 1000, 1e-7, 1e-3, 0, 1e-5, 1e-5, 0]        # testBFGS params (Source/Examples.cpp:247); [7] = maxIter
SW = [1e-4, 0.8, 1e-6, 1.0, 1e-10, 2.0, 50, 1e-5, 1e-6, 1e-3, 0, 1e-5, 1e-5, 0]     # testBFGSBndMPISW params (:37); [10] = maxIter


def _run(lib_bfgs, variant, obj, x0, iters):
    if variant == "bfgs":
        p = list(BF)
        p[7] = iters
        return lib_bfgs(variant, obj, x0, p)
    p = list(SW)
    p[10] = iters
    return lib_bfgs(variant, obj, x0, p, np.full(x0.size, -5.0), np.full(x0.size, 5.0), pool=8)


@pytest.mark.parametrize("variant", ["bfgs", "bfgs_bnd_sw"])
@pytest.mark.parametrize("obj,x0,xopt", [("rosenbrock", np.full(10, 3.0), np.ones(10)), ("booth", np.array([3.0, -2.0]), np.array([1.0, 3.0]))])
def test_bfgs_reaches_the_optimum_with_analytic_gradients(host, variant, obj, x0, xopt):
    def call(v, o, x, p, lb=None, ub=None, pool=0):
        return host.bfgs(v, o, x, p, lb, ub, pool_width=pool)
    r = _run(call, variant, obj, x0, 1000)
    # the stop tests of both classes are ||x_k+1 - x_k|| < xMinDiff (1e-5) or ||g|| < minGrad2Norm (1e-5): within 1e-4 of the optimum
    assert np.linalg.norm(r["X"] - xopt) <= 1e-4 * np.linalg.norm(xopt), (r["X"], r["iterations"])
    assert r["fOpt"] < 1e-8


@pytest.mark.parametrize("variant,obj,x0,iters", [("bfgs", "rosenbrock", np.full(10, 3.0), 5), ("bfgs", "booth", np.array([3.0, -2.0]), 5),
                                                  ("bfgs_bnd_sw", "rosenbrock", np.full(10, 3.0), 5),
                                                  ("bfgs_bnd_sw", "booth", np.array([3.0, -2.0]), 3)])
def test_bfgs_iterates_match_the_host_logic_stand_in(host, variant, obj, x0, iters):
    """The stand-in runs the same host controllers with the partials and the dense algebra on the CPU, in the literal two-product
    updateHessianInv; the GPU is set to the same form. What remains is the summation order of the device's dense algebra."""
    import test_host_logic_cpu as TH
    hl = HLG.build_and_load()
    if hl is None:
        pytest.skip("no g++ on this box")
    host.set_hinv_mode(capi.HINV_LITERAL)
    hl.pnolhost_set_analytic_gradient(1)
    try:
        def gpu(v, o, x, p, lb=None, ub=None, pool=0):
            return host.bfgs(v, o, x, p, lb, ub, pool_width=pool)

        def cpu(v, o, x, p, lb=None, ub=None, pool=0):
            return TH.bfgs(hl, v, o, x, p, lb, ub, pool=pool)
        a, b = _run(gpu, variant, obj, x0, iters), _run(cpu, variant, obj, x0, iters)
    finally:
        hl.pnolhost_set_analytic_gradient(0)
    assert a["iterations"] == b["iterations"]
    assert np.linalg.norm(a["X"] - b["X"]) <= 1e-9 * np.linalg.norm(b["X"]), (a["X"], b["X"])
    assert abs(a["fOpt"] - b["fOpt"]) <= 1e-9 * max(abs(b["fOpt"]), 1e-300) or a["fOpt"] == b["fOpt"]


# ---- column split over several GPUs ----
def _ngpu():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    from parallelnonlinearoptimizationlibrary_b200 import capi as K, hostapi, launch
    launch.init_process_group("nccl")
    ctx = K.Context(rank)
    assert launch.attach_communicator(ctx) == world
    f = ctx.functor(K.F_ROSENBROCK)
    hostapi.attach(ctx)
    hostapi.set_analytic_gradient(True)
    for n in (40, 4096):
        x = np.random.default_rng(n).uniform(-2, 2, n)
        g, f0 = ctx.gradient(f, x, want_f0=True)
        gm = hostapi.gradient("rosenbrock", x, np.full(n, 1e-7), mpi=True)     # gradientApproximationMPI: the sharded call
        np.save(os.path.join(out_dir, "g%d_%d.npy" % (n, rank)), np.concatenate([g, [f0], gm]))
    hostapi.set_analytic_gradient(False)
    hostapi.detach()
    launch.barrier()
    f.close()
    ctx.close()
    import torch.distributed as dist
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 4, 8])
def test_sharded_gradient_is_the_single_gpu_gradient(ctx, tmp_path, world):
    if _ngpu() < world:
        pytest.skip("needs %d GPUs" % world)
    import socket
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    mp.spawn(_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    f = ctx.functor(capi.F_ROSENBROCK)
    for n in (40, 4096):
        x = np.random.default_rng(n).uniform(-2, 2, n)
        g, f0 = ctx.gradient(f, x, want_f0=True)
        want = np.concatenate([g, [f0], g])
        for r in range(world):
            assert np.array_equal(np.load(tmp_path / ("g%d_%d.npy" % (n, r))), want), (n, r)
    f.close()
