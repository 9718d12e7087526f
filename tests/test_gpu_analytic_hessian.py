"""GPU: analytic Hessians (pnol_hessian) against the host definition of every partial2 (include/pnol/functors.hpp, the user's
tests/user_functor/my_hessians.hpp) bit for bit, up to the largest n that fits; the refusals; the plugin member and the BFGS classes with
initHessFD and Runtime::setAnalyticHessian(true), against the same controllers run on the CPU stand-in extended by the host partial2()
(tests/host_logic_standin.cpp); and every rank of a communicator returning the one-GPU bits."""
import os
import sys

import numpy as np
import pytest

import host_standin
import test_user_hessian_cpu as HC
import user_functor_lib as UF
import user_gradient_lib as UG
import user_hessian_lib as UH
from parallelnonlinearoptimizationlibrary_b200 import capi

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _nmax():
    """(opt-in shared memory - one 32 x 33 tile) / 8 bytes: 28000 on a B200"""
    import torch
    return (int(torch.cuda.get_device_properties(0).shared_memory_per_block_optin) - 32 * 33 * 8) // 8


def _t_y():
    t = np.linspace(-2.0, 3.0, 257)
    return t, 1.5 * np.exp(0.7 * t) + 0.2 + 0.01 * np.sin(7 * t)


# kind, scalars, ints, columns, smallest n, start-point scale; columns "A": the quadratic form's n x n matrix (built per n)
CASES = {
    "rosenbrock": (capi.F_ROSENBROCK, (), (), (), 1, 2.0),
    "power3": (capi.F_POWER, (), (3,), (), 1, 2.0),
    "booth": (capi.F_BOOTH, (), (), (), 2, 3.0),
    "goldstein": (capi.F_GOLDSTEIN, (), (), (), 2, 2.0),
    "rastrigin": (capi.F_RASTRIGIN, (), (), (), 1, 5.12),
    "expsingle": (capi.F_EXPCURVE_SINGLE, (), (), _t_y(), 3, 1.0),
    "user_styblinski": (UH.MYH_F_STYBLINSKI, (0.5,), (), (), 1, 4.0),
    "user_quadform": (UH.MYH_F_QUADFORM, (), (), "A", 1, 1.0),
}
SPARSE = ["rosenbrock", "power3", "booth", "goldstein", "rastrigin", "expsingle", "user_styblinski"]
NS = [1, 2, 3, 31, 32, 33, 64, 1000, 4096]


@pytest.fixture(scope="module")
def user():
    return UH.build_and_load()


def _columns(name, n):
    cols = CASES[name][3]
    if cols == "A":
        return (np.random.default_rng(n + 1).normal(size=n * n),)
    return cols


def _functor(ctx, name, cols):
    kind, sc, ints, _, _, _ = CASES[name]
    m = 0 if not cols else (cols[0].numel() if hasattr(cols[0], "numel") else cols[0].size)
    return ctx.functor(kind, sc, ints, cols, m)


def _host(name, x, cols):
    kind, sc, ints, _, _, _ = CASES[name]
    return UH.host_hessian(kind, x, sc, ints, cols)


def _bits(a):
    return np.ascontiguousarray(a).view(np.int64)


@pytest.mark.parametrize("name", sorted(CASES))
def test_hessian_is_the_host_partial2_bit_for_bit(ctx, user, name):
    import torch
    nmin, scale = CASES[name][4], CASES[name][5]
    rng = np.random.default_rng(len(name))
    for n in NS:
        if n < nmin:
            continue
        x = rng.uniform(-scale, scale, n)
        cols = _columns(name, n)
        f = _functor(ctx, name, cols)
        want = _host(name, x, cols)
        H = ctx.hessian(f, x)
        assert np.array_equal(_bits(H), _bits(want)), (name, n)
        if n in (33, 4096):
            # device pointers, x misaligned by one double, H prefilled with NaN (every entry is written), symmetric bit for bit
            xb = torch.empty(n + 1, dtype=torch.float64, device="cuda")
            xb[1:] = torch.from_numpy(x).cuda()
            Hd = torch.full((n, n), float("nan"), dtype=torch.float64, device="cuda")
            torch.cuda.synchronize()
            ctx.hessian(f, xb.data_ptr() + 8, H=Hd.data_ptr(), n=n)
            assert torch.equal(Hd, Hd.T), (name, n)
            assert np.array_equal(_bits(Hd.cpu().numpy()), _bits(want)), (name, n)
        f.close()


def _band(n):
    """(i, j), i <= j: the diagonal, the first super-diagonal and the leading 3 x 3 block"""
    ii = np.concatenate([np.arange(n), np.arange(n - 1), [0, 0, 1]])
    jj = np.concatenate([np.arange(n), np.arange(1, n), [1, 2, 2]])
    key = np.unique(ii.astype(np.int64) * n + jj)
    return (key // n).astype(np.int32), (key % n).astype(np.int32)


@pytest.mark.parametrize("name", SPARSE)
def test_hessian_at_the_largest_n_is_the_host_band_and_plus_zero_elsewhere(ctx, user, name):
    import torch
    n = _nmax()
    x = np.random.default_rng(n).uniform(-CASES[name][5], CASES[name][5], n)
    cols = _columns(name, n)
    f = _functor(ctx, name, cols)
    xd = torch.from_numpy(x).cuda()
    H = torch.full((n, n), float("nan"), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    ctx.hessian(f, xd, H=H, n=n)
    ii, jj = _band(n)
    kind, sc, ints = CASES[name][:3]
    want = UH.host_partial2(kind, x, ii, jj, sc, ints, cols)
    ti, tj = torch.from_numpy(ii.astype(np.int64)).cuda(), torch.from_numpy(jj.astype(np.int64)).cuda()
    upper, lower = H[ti, tj].cpu().numpy(), H[tj, ti].cpu().numpy()
    assert np.array_equal(_bits(upper), _bits(want)) and np.array_equal(_bits(lower), _bits(want)), name
    # every entry outside the band (both triangles) is +0: count the entries whose bits are not those of +0
    Hb = H.view(torch.int64)
    nonzero = int((Hb != 0).sum())
    off = np.where(ii == jj, 1, 2)
    assert nonzero == int(np.sum(off * (_bits(want) != 0))), name
    assert torch.equal(Hb, Hb.T)
    del H, Hb
    f.close()


def test_quadratic_form_is_the_host_partial2_up_to_n_8192(ctx, user):
    import torch
    for n in (4097, 8192):
        A = np.random.default_rng(n).normal(size=n * n)
        x = np.random.default_rng(n + 1).uniform(-1, 1, n)
        Ad = torch.from_numpy(A).cuda()          # a device column is borrowed, not copied
        f = _functor(ctx, "user_quadform", (Ad,))
        H = torch.full((n, n), float("nan"), dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        ctx.hessian(f, torch.from_numpy(x).cuda(), H=H, n=n)
        assert np.array_equal(_bits(H.cpu().numpy()), _bits(_host("user_quadform", x, (A,)))), n
        f.close()


def test_functors_without_a_second_derivative_and_bad_calls_are_refused(ctx, user):
    import torch
    lib = ctx.lib
    UF.build_and_load()
    UG.build_and_load()
    x, H = np.full(4, 0.5), np.empty(16)
    # user scalar objectives without partial2() -- Trid with partial() only, Trid without any derivative: refused, never a forward
    # difference; the error names the kind
    for kind in (UG.MYG_F_TRID, UF.MY_F_TRID):
        ft = ctx.functor(kind)
        assert lib.pnol_hessian(ctx.h, ft.handle, capi._ptr(x), 4, capi._ptr(H)) == capi.ERR_NO_FUNCTOR
        assert str(kind).encode() in lib.pnol_last_error(ctx.h) and b"partial2" in lib.pnol_last_error(ctx.h)
        ft.close()
    # residual models: refused as the forward difference refuses them
    t, y = _t_y()
    for fr in (ctx.functor(capi.F_EXPCURVE, (), (), (t, y), t.size), ctx.functor(UF.MY_F_GAUSSFIT, (0.3,), (), (t, y), t.size)):
        st = lib.pnol_hessian(ctx.h, fr.handle, capi._ptr(x[:3]), 3, capi._ptr(H))
        st_fd = lib.pnol_fd_hessian(ctx.h, fr.handle, capi._ptr(x[:3]), capi._ptr(np.full(3, 1e-4)), 3, capi._ptr(H))
        assert st == st_fd != capi.PNOL_OK
        fr.close()
    # one coordinate more than the point and a tile leave room for in shared memory (device buffers: nothing is staged)
    fr = ctx.functor(capi.F_ROSENBROCK)
    n = _nmax() + 1
    xd = torch.full((n,), 0.5, dtype=torch.float64, device="cuda")
    Hd = torch.empty(1, dtype=torch.float64, device="cuda")
    assert lib.pnol_hessian(ctx.h, fr.handle, capi._ptr(xd), n, capi._ptr(Hd)) == capi.ERR_INVALID
    assert ("n = %d is outside 1 .. %d" % (n, n - 1)).encode() in lib.pnol_last_error(ctx.h)
    # bad arguments
    assert lib.pnol_hessian(ctx.h, fr.handle, capi._ptr(x), 0, capi._ptr(H)) == capi.ERR_INVALID
    assert lib.pnol_hessian(ctx.h, fr.handle, None, 4, capi._ptr(H)) == capi.ERR_INVALID
    assert lib.pnol_hessian(ctx.h, fr.handle, capi._ptr(x), 4, None) == capi.ERR_INVALID
    fr.close()


# ---- the plugin classes ----
@pytest.fixture
def host(ctx):
    from parallelnonlinearoptimizationlibrary_b200 import hostapi
    hostapi.attach(ctx)
    yield hostapi
    hostapi.set_analytic_gradient(False)
    hostapi.set_analytic_hessian(False)
    hostapi.set_hinv_mode(capi.HINV_RANK2)
    hostapi.detach()


@pytest.mark.parametrize("obj,name,n", [("rosenbrock", "rosenbrock", 40), ("booth", "booth", 2), ("goldstein", "goldstein", 2),
                                        ("power:3", "power3", 5), ("rastrigin", "rastrigin", 12)])
def test_objective_member_returns_the_pnol_hessian_bits(ctx, host, obj, name, n):
    x = np.random.default_rng(n).uniform(-1.5, 1.5, n)
    f = _functor(ctx, name, ())
    dx = np.full(n, 1e-4)
    assert np.array_equal(_bits(host.hessian(obj, x, dx)), _bits(ctx.fd_hessian(f, x, dx)))       # switch off: the forward difference
    host.set_analytic_hessian(True)
    want = ctx.hessian(f, x)
    assert np.array_equal(_bits(host.hessian(obj, x, np.full(n, np.nan))), _bits(want))             # dX is not read
    f.close()


@pytest.mark.parametrize("variant", sorted(HC.VARIANTS))
def test_bfgs_with_analytic_initial_hessian_reaches_the_optimum(host, variant):
    host.set_analytic_gradient(True)
    host.set_analytic_hessian(True)

    def call(v, o, x, p, lb, ub, pool):
        return host.bfgs(v, o, x, p, lb, ub, pool_width=pool)
    for obj, x0, xopt, fopt in HC.PROBLEMS:
        if obj == "rosenbrock" and variant in ("bfgs_mpi", "bfgsbnd_mpi"):
            continue            # these two stop short of the optimum from this start with the forward-difference Hessian too
        r = HC.run_bfgs(call, variant, obj, x0, 1000)
        assert np.linalg.norm(r["X"] - xopt) <= 1e-4 * max(np.linalg.norm(xopt), 1.0), (obj, r)
        assert abs(r["fOpt"] - fopt) < 1e-8, (obj, r)


@pytest.mark.parametrize("variant", sorted(HC.VARIANTS))
@pytest.mark.parametrize("obj", ["rosenbrock", "booth", "goldstein"])
def test_bfgs_iterates_match_the_host_logic_stand_in(host, variant, obj):
    """initHessFD = 1 with analytic gradient and Hessian. The stand-in runs the same host controllers with the host partials, the host
    partial2 and the dense algebra on the CPU (LU inverse included), in the literal two-product updateHessianInv; the GPU is set to the
    same form. What remains is the summation order of the device's dense algebra."""
    import test_host_logic_cpu as TH
    hl = host_standin.load()
    if hl is None:
        pytest.skip("no g++ on this box")
    x0 = {p[0]: p[1] for p in HC.PROBLEMS}[obj]
    # Booth is a quadratic: from the exact inverse Hessian the first step lands on the optimum up to rounding, and the steps after it
    # follow the rounding of a gradient near 0 (BFGSBnd_MPI then wanders by 4e-4 either way) -- compare that first step
    iters = 1 if obj == "booth" else 5
    host.set_hinv_mode(capi.HINV_LITERAL)
    host.set_analytic_gradient(True)
    host.set_analytic_hessian(True)
    hl.pnolhost_set_analytic_gradient(1)
    hl.pnolhost_set_analytic_hessian(1)
    try:
        a = HC.run_bfgs(lambda v, o, x, p, lb, ub, pool: host.bfgs(v, o, x, p, lb, ub, pool_width=pool), variant, obj, x0, iters)
        b = HC.run_bfgs(lambda v, o, x, p, lb, ub, pool: TH.bfgs(hl, v, o, x, p, lb, ub, pool), variant, obj, x0, iters)
    finally:
        hl.pnolhost_set_analytic_gradient(0)
        hl.pnolhost_set_analytic_hessian(0)
    assert a["iterations"] == b["iterations"]
    assert np.linalg.norm(a["X"] - b["X"]) <= 1e-9 * np.linalg.norm(b["X"]), (a["X"], b["X"])
    assert abs(a["fOpt"] - b["fOpt"]) <= 1e-9 * max(abs(b["fOpt"]), 1e-300) or a["fOpt"] == b["fOpt"]


# ---- a communicator attached: no collective, every rank the whole matrix ----
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
    hostapi.set_analytic_hessian(True)
    for n in (40, 1000):
        x = np.random.default_rng(n).uniform(-2, 2, n)
        H = ctx.hessian(f, x)
        Hm = hostapi.hessian("rosenbrock", x, np.full(n, np.nan))
        np.save(os.path.join(out_dir, "H%d_%d.npy" % (n, rank)), np.stack([H, Hm]))
    hostapi.set_analytic_hessian(False)
    hostapi.detach()
    launch.barrier()
    f.close()
    ctx.close()
    import torch.distributed as dist
    dist.destroy_process_group()


def test_every_rank_of_a_communicator_returns_the_single_gpu_hessian(ctx, tmp_path):
    world = 2
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
    for n in (40, 1000):
        H = ctx.hessian(f, np.random.default_rng(n).uniform(-2, 2, n))
        for r in range(world):
            got = np.load(tmp_path / ("H%d_%d.npy" % (n, r)))
            assert np.array_equal(_bits(got), _bits(np.stack([H, H]))), (n, r)
    f.close()
