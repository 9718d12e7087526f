"""CPU: the host controllers of the plugin API (parallelnonlinearoptimizationlibrary_b200/host/*.cpp: BFGS, BFGS_MPI, BFGS_Bnd,
BFGS_Bnd_MPI_SW, BFGSBnd_MPI, SimplexSearch, LevMarq, LevMarqMPI, GeneticAlgorithm[MPI], the Objective stencil members, the box helpers)
WITHOUT a GPU: the unmodified host sources
are linked into a test-only library against oracle/host_logic_device.cpp, which answers the C-ABI calls of these paths with the CPU
oracle instead of CUDA kernels (test infrastructure; the product libraries have no CPU path and this library is never shipped).

With the oracle's arithmetic underneath -- the same sequential sums and literal two-product updateHessianInv the verbatim reference
was compiled with -- every controller reproduces the committed outputs of the verbatim reference BIT FOR BIT: iterates, f0, fOpt,
iteration counts, random draws. So the control flow (line searches, pools, active-set recursion, steepest-descent retries, Nelder-Mead
steps, and the accept / reject / damping rule of Levenberg-Marquardt with and without a stored Jacobian) is the reference's, decision
for decision, and what the GPU tests see beyond that (1e-9 ... 1e-5, tests/test_gpu_host_api.py)
is the summation order of the device's dense algebra and nothing else."""
import ctypes as C
import glob
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

import host_standin

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(HERE, "golden"))

G = np.load(os.path.join(HERE, "golden", "ref_golden.npz"))


def g(case, name):
    return G["%s/%s" % (case, name)]


@pytest.fixture(scope="module")
def hl():
    so = host_standin.base_path()
    if so is None:
        pytest.skip("no g++ on this box")
    lib = C.CDLL(so, mode=C.RTLD_LOCAL)
    lib.pnolhost_last_error.restype = C.c_char_p
    lib.pnolhost_set_hinv_mode(0)          # PNOL_HINV_LITERAL: the reference's two matrix products
    return lib


def _p(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def bfgs(lib, variant, obj, x0, params, lb=None, ub=None, pool=0):
    X = np.array(x0, dtype=np.float64).copy()
    p = np.array(params, dtype=np.float64)
    lb = None if lb is None else np.ascontiguousarray(lb, dtype=np.float64)
    ub = None if ub is None else np.ascontiguousarray(ub, dtype=np.float64)
    f0, fo, it = C.c_double(), C.c_double(), C.c_int()
    st = lib.pnolhost_bfgs(variant.encode(), obj.encode(), _p(X), X.size, _p(p), _p(lb), _p(ub), int(pool), 0, C.byref(f0), C.byref(fo), C.byref(it))
    assert st == 0, (st, lib.pnolhost_last_error())
    return dict(X=X, f0=f0.value, fOpt=fo.value, iterations=it.value)


def same(r, case):
    return np.array_equal(r["X"], g(case, "X")) and r["f0"] == g(case, "f0")[0] and r["fOpt"] == g(case, "fOpt")[0]


BF = [1e-4, 0.9, 1e-6, 1.0, 1000, 1e-7, 1e-3, 0, 1e-5, 1e-5, 0]        # testBFGS params (Source/Examples.cpp:247); [7] = maxIter
SW = [1e-4, 0.8, 1e-6, 1.0, 1e-10, 2.0, 50, 1e-5, 1e-6, 1e-3, 0, 1e-5, 1e-5, 0]     # testBFGSBndMPISW params (:37); [10] = maxIter


@pytest.mark.parametrize("case,n,x0,iters", [("bfgs_cfg1_it5", 10, 3.0, 5), ("bfgs_cfg1_it100", 10, 3.0, 100), ("testBFGS", 5, 3.0, 100)])
def test_bfgs_bit_for_bit(hl, case, n, x0, iters):
    p = list(BF)
    p[7] = iters
    assert same(bfgs(hl, "bfgs", "rosenbrock", np.full(n, x0), p), case)


@pytest.mark.parametrize("iters", [5, 60])
def test_bfgs_mpi_pool_bit_for_bit(hl, iters):
    p = [1e-4, 0.9, 4.0, 1.0, 50, 1e-7, 1e-3, iters, 1e-5, 1e-5, 0]
    assert same(bfgs(hl, "bfgs_mpi", "rosenbrock", np.full(10, 10.0), p, pool=4), "bfgs_mpi_P4_it%d" % iters)


@pytest.mark.parametrize("case,P,iters", [("testBFGSBndMPISW_P2", 2, 200), ("testBFGSBndMPISW_P8", 8, 200), ("bfgs_bnd_sw_n64_P8_it3", 8, 3),
                                          ("bfgs_bnd_sw_n64_P8_it20", 8, 20)])
def test_bfgs_bnd_mpi_sw_bit_for_bit(hl, case, P, iters):
    p = list(SW)
    p[10] = iters
    x0 = g(case, "x0")
    lb, ub = (g(case, "lb"), g(case, "ub")) if case.startswith("test") else (np.full(x0.size, -5.0), np.full(x0.size, 5.0))
    assert same(bfgs(hl, "bfgs_bnd_sw", "rosenbrock", x0, p, lb, ub, pool=P), case)


@pytest.mark.parametrize("case,n,iters", [("testBFGSBnd_it4", 5, 4), ("testBFGSBnd_it200", 5, 200), ("bfgs_bnd_n12_it6", 12, 6)])
def test_bfgs_bnd_serial_bit_for_bit(hl, case, n, iters):
    p = list(SW)
    p[10] = iters
    x0 = g(case, "x0") if case.startswith("bfgs_bnd") else np.full(n, 2.0)
    assert same(bfgs(hl, "bfgs_bnd", "rosenbrock", x0, p, np.full(n, -5.0), np.full(n, 5.0)), case)


def test_bfgsbnd_mpi_bit_for_bit(hl):
    from make_bfgsbnd_mpi_golden import PARAMS, cases
    G2 = np.load(os.path.join(HERE, "golden", "bfgsbnd_mpi_golden.npz"))
    k = PARAMS
    for name, (obj, x0, lb, ub, P, iters, extra, _) in cases().items():
        p = [k["c1"], k["c2"], k["alphamin"], k["maxalphamult"], k["alphaguess"], k["maxiterls"], k["dxgrad"], k["dxhess"], iters, k["xmindiff"],
             k["mingrad"], k["fsteptol"], extra.get("inithess", 0)]
        r = bfgs(hl, "bfgsbnd_mpi", obj, x0, p, lb, ub, pool=P)
        assert np.array_equal(r["X"], G2[name + "/X"]) and r["f0"] == G2[name + "/f0"][0] and r["fOpt"] == G2[name + "/fOpt"][0], name
        assert r["iterations"] == int(G2[name + "/iterations_done"]), name       # outer + recursive iterations


def test_simplex_search_bit_for_bit(hl):
    from make_simplex_golden import CASES
    S = np.load(os.path.join(HERE, "golden", "simplex_golden.npz"))
    for name, (obj, x0, kw, stream) in CASES.items():
        if stream[0] == "values":
            vals = np.ascontiguousarray(stream[1], dtype=np.float64)
            hl.pnolhost_set_stream(_p(vals), C.c_ulonglong(vals.size), C.c_ulonglong(0), C.c_double(1.0))
        else:
            hl.pnolhost_set_stream(C.c_void_p(0), C.c_ulonglong(0), C.c_ulonglong(stream[1]), C.c_double(stream[2]))
        X = np.array(x0, dtype=np.float64).copy()
        p = np.array([kw.get("alpha", 1.0), kw.get("gamma", 2.0), kw.get("rho", 0.5), kw.get("sigma", 0.5), kw.get("maxiter", 10000),
                      kw.get("initrandmax", 1.0), kw.get("xmindiff", 1e-7)], dtype=np.float64)
        f0, fo = C.c_double(), C.c_double()
        rep = np.zeros(2)
        try:
            st = hl.pnolhost_simplex(obj.encode(), _p(X), X.size, _p(p), 0, C.byref(f0), C.byref(fo), _p(rep))
        finally:
            hl.pnolhost_clear_stream()
        assert st == 0, hl.pnolhost_last_error()
        assert np.array_equal(X, S[name + "/X"]) and f0.value == S[name + "/f0"][0] and fo.value == S[name + "/fOpt"][0], name
        assert int(rep[1]) == int(S[name + "/stream_pos"][0])


@pytest.mark.parametrize("case", ["lm_lorentz_K8", "lm_lorentz_K16"])
@pytest.mark.parametrize("serial", [0, 1])
@pytest.mark.parametrize("store_j", [1, 0])
@pytest.mark.parametrize("whole_loop_call", [0, 1])
def test_levenberg_marquardt_bit_for_bit(hl, case, serial, store_j, whole_loop_call):
    # LevMarqMPI / LevMarq::findMin (accept / reject, damping, stop rule on the host; residuals, FD Jacobian, normal equations and solve
    # behind pnol_residual_eval / pnol_lm_step), with a J buffer and without one (Runtime::setStoreJacobian(false)); whole_loop_call:
    # with the Jacobian cache off findMin hands its while loop to pnol_lm_iterate in one call
    t, y, w, x0, iters = g(case, "t"), g(case, "y"), float(g(case, "w")), g(case, "x0"), int(g(case, "iters"))
    hl.pnolhost_set_store_jacobian(store_j)
    hl.pnolhost_set_jacobian_cache(0 if whole_loop_call else 1)
    try:
        X = x0.copy()
        m = t.size
        F0, F, rep = np.empty(m), np.empty(m), np.zeros(6)
        st = hl.pnolhost_lm_lorentz(_p(t), _p(y), C.c_longlong(m), C.c_double(w), _p(X), X.size, C.c_double(0.001), C.c_double(10.0),
                                    C.c_double(1e-7), C.c_double(iters), C.c_double(0.0), serial, _p(F0), _p(F), _p(rep))
    finally:
        hl.pnolhost_set_store_jacobian(1)
        hl.pnolhost_set_jacobian_cache(1)
    assert st == 0, hl.pnolhost_last_error()
    assert np.array_equal(X, g(case, "X")) and np.array_equal(F0, g(case, "F0")) and np.array_equal(F, g(case, "F"))
    assert int(rep[0]) == iters and int(rep[1]) + int(rep[2]) == iters          # iterations = accepted + rejected


def test_levenberg_marquardt_reference_examples(hl):
    # testLMCubicLinearCoef (Source/Examples.cpp:415-452): bit for bit. testLMExpMPI (:128-159): the product's ExpCurve model calls the
    # shared host/device exp instead of libm's (include/pnol/ExampleObjectives.hpp), so the fit agrees to 1e-9, not to the bit
    for name, key, x0, exact in (("cubic", "testLMCubicLinearCoef", np.full(4, 0.1), True), ("expcurve", "testLMExpMPI", np.array([9.0, 0.5, 0.3]), False)):
        X = x0.copy()
        rep = np.zeros(6)
        st = hl.pnolhost_lm_example(name.encode(), _p(X), X.size, C.c_double(0.001), C.c_double(10.0), C.c_double(1e-6), C.c_double(100.0),
                                    C.c_double(1e-6), None, None, _p(rep))
        assert st == 0, hl.pnolhost_last_error()
        if exact:
            assert np.array_equal(X, g(key, "X"))
        else:
            assert np.linalg.norm(X - g(key, "X")) <= 1e-9 * np.linalg.norm(g(key, "X"))
            assert np.allclose(X, [10.2, 0.4, 0.1], rtol=1e-8)              # the known answer (Source/ExampleObjectives.hpp:145)


@pytest.mark.parametrize("spec,obj", [("powerprod2", "power:2"), ("rastrigin", "rastrigin"), ("rosenbrock", "rosenbrock")])
@pytest.mark.parametrize("serial", [0, 1])
def test_genetic_algorithm_host_class_bit_for_bit(hl, spec, obj, serial):
    # GeneticAlgorithmMPI / GeneticAlgorithm::findMinBnd over the GA state machine of the C-ABI (answered by replaying the oracle's
    # restatement of the loop): result, f0, fOpt, generations and the number of random draws of the verbatim reference
    c = "ga_%s" % spec
    hl.pnolhost_set_stream(C.c_void_p(0), C.c_ulonglong(0), C.c_ulonglong(int(g(c, "seed"))), C.c_double(float(g(c, "scale"))))
    X = g(c, "x0").copy()
    lb, ub = g(c, "lb"), g(c, "ub")
    f0, fo = C.c_double(), C.c_double()
    rep = np.zeros(7)
    try:
        st = hl.pnolhost_ga(obj.encode(), _p(X), X.size, _p(lb), _p(ub), int(g(c, "npop")), int(g(c, "gens")), C.c_double(0.1), C.c_double(0.3),
                            C.c_double(0.2), C.c_double(0.5), C.c_double(0.01), C.c_double(50.0), serial, C.byref(f0), C.byref(fo), _p(rep))
    finally:
        hl.pnolhost_clear_stream()
    assert st == 0, hl.pnolhost_last_error()
    assert np.array_equal(X, g(c, "X")) and f0.value == g(c, "f0")[0] and fo.value == g(c, "fOpt")[0]
    assert int(rep[0]) == int(g(c, "gens")) and int(rep[2]) == int(g(c, "stream_pos")[0])


@pytest.mark.parametrize("spec,obj,n", [("rosenbrock", "rosenbrock", 5), ("rosenbrock", "rosenbrock", 40), ("booth", "booth", 2),
                                        ("goldstein", "goldstein", 2), ("powerprod3", "power:3", 5), ("rastrigin", "rastrigin", 12)])
def test_objective_stencil_members_bit_for_bit(hl, spec, obj, n):
    # Objective::gradientApproximation / gradientApproximationMPI / hessianApproximation as a user calls them, against the committed
    # outputs of the reference's own members (Source/PNOL_Objective.cpp:12-34, 88-159, 38-85)
    case = "fdgrad_%s_%d" % (spec, n)
    x, dx = np.ascontiguousarray(g(case, "x")), np.ascontiguousarray(g(case, "dx"))
    for which, key in ((0, "g"), (1, "g_mpi")):
        out = np.empty(n)
        assert hl.pnolhost_gradient(obj.encode(), _p(x), _p(dx), n, which, _p(out)) == 0, hl.pnolhost_last_error()
        assert np.array_equal(out, g(case, key))
    if n <= 12:
        dxh = np.ascontiguousarray(g(case, "dxh"))
        B = np.empty((n, n))
        assert hl.pnolhost_hessian(obj.encode(), _p(x), _p(dxh), n, _p(B)) == 0, hl.pnolhost_last_error()
        assert np.array_equal(B, g(case, "B"))


def test_recur_gradient_and_box_helpers_bit_for_bit(hl):
    c = "recur_rosenbrock_8"
    xr, constx = np.ascontiguousarray(g(c, "xr")), np.ascontiguousarray(g(c, "constx"))
    ind = np.ascontiguousarray(g(c, "ind"), dtype=np.uint8)
    dxr = np.full(xr.size, 1e-6)
    gr, f = np.empty(xr.size), C.c_double()
    assert hl.pnolhost_gradient_recur(b"rosenbrock", _p(xr), _p(dxr), xr.size, _p(constx), _p(ind), constx.size, _p(gr), C.byref(f)) == 0
    assert np.array_equal(gr, g(c, "g_mpi")) and f.value == g(c, "f")[0]
    hl.pnolhost_compute_alpha_bnd.restype = C.c_double
    x, lb, ub, p = (np.ascontiguousarray(g("box", k)) for k in ("xin", "lb", "ub", "p"))
    assert hl.pnolhost_compute_alpha_bnd(_p(x), _p(lb), _p(ub), _p(p), x.size) == g("box", "alphabnd")[0]
    xo = np.ascontiguousarray(g("box", "x")).copy()
    assert hl.pnolhost_check_box_bounds(_p(xo), _p(lb), _p(ub), xo.size) == 0
    assert np.array_equal(xo, g("box", "Xfixed"))


def test_paths_outside_the_stand_in_fail_loudly(hl):
    # what the stand-in does not answer comes back as an error through the host classes, nothing is faked: invalid GA fractions, and a
    # residual model handed to a scalar algorithm
    X = np.full(4, 3.0)
    lb, ub = np.full(4, -10.0), np.full(4, 10.0)
    f0, fo = C.c_double(), C.c_double()
    rep = np.zeros(7)
    hl.pnolhost_set_stream(C.c_void_p(0), C.c_ulonglong(0), C.c_ulonglong(1), C.c_double(0.99))
    try:
        st = hl.pnolhost_ga(b"rosenbrock", _p(X), 4, _p(lb), _p(ub), 50, 3, C.c_double(0.6), C.c_double(0.6), C.c_double(0.2), C.c_double(0.5),
                            C.c_double(0.01), C.c_double(50.0), 0, C.byref(f0), C.byref(fo), _p(rep))
    finally:
        hl.pnolhost_clear_stream()
    assert st != 0 and b"random children" in hl.pnolhost_last_error()
    st = hl.pnolhost_bfgs(b"bfgs", b"no_such_objective", _p(X), 4, _p(np.zeros(11)), None, None, 0, 0, C.byref(f0), C.byref(fo), C.byref(C.c_int()))
    assert st != 0


def test_reference_example_drivers_print_the_reference_numbers(tmp_path):
    # The reference's OWN Source/Examples.cpp (unmodified, from where it lies; oracle/dropin_examples.cpp) compiled against include/pnol,
    # the unmodified host sources and the oracle-backed stand-in: what its drivers print is what the verbatim reference prints
    # (tests/golden/examples_ref.json) -- iterates digit for digit (17 significant digits) and, for the serial classes, the number of
    # objective evaluations (getEvals(): host objEval calls + points evaluated behind the C-ABI). Needs /root/reference to build.
    import json
    from test_gpu_dropin_examples import scalar, vectors
    cxx = shutil.which("g++")
    if cxx is None or not os.path.isdir("/root/reference/Source"):
        pytest.skip("needs g++ and /root/reference (the reference's Examples.cpp is compiled from where it lies)")
    host = os.path.join(ROOT, "parallelnonlinearoptimizationlibrary_b200", "host")
    exe = str(tmp_path / "examples_cpu")
    inc = os.path.join(ROOT, "include")
    subprocess.check_call([cxx, "-std=c++17", "-O2", "-ffp-contract=off", "-w", "-I" + os.path.join(inc, "pnol", "nompi"), "-I" + os.path.join(inc, "pnol"),
                           "-I" + inc, "-I" + host, "-I/root/reference/Source", os.path.join(ROOT, "oracle", "dropin_examples.cpp")] +
                          sorted(glob.glob(os.path.join(host, "*.cpp"))) +
                          [os.path.join(ROOT, "oracle", "host_logic_device.cpp"), os.path.join(ROOT, "oracle", "pnol_oracle.cpp"), "-o", exe])
    ref = json.load(open(os.path.join(HERE, "golden", "examples_ref.json")))

    def run(driver):
        r = subprocess.run([exe, driver, str(ref["pool_width"]), str(ref["seed"])], capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, (driver, r.stderr[-500:])
        return r.stdout, ref["tails"][driver]

    for driver, key in (("testBFGS", "X = "), ("testBFGS_booth", "X = "), ("testBFGS_MPI", "X = "), ("testBFGSBnd", "Xopt = "),
                        ("testBFGSBndMPISW", "Xopt = "), ("testBFGSBnd_MPI", "X = ")):
        ours, want = run(driver)
        assert np.array_equal(vectors(ours, key)[-1], vectors(want, key)[-1]), driver
        assert scalar(ours, "f0 =") == scalar(want, "f0 =")
    for driver in ("testBFGS", "testBFGS_booth", "testBFGSBnd"):                 # serial classes: same evaluation count
        ours, want = run(driver)
        assert scalar(ours, "Optimization used") == scalar(want, "Optimization used"), driver
    ours, want = run("testSimplexSearch")
    assert scalar(ours, "Optimization used") == scalar(want, "Optimization used") == 3884
    assert np.allclose(vectors(ours, "X = ")[-1], vectors(want, "X = ")[-1], atol=2e-5)      # the reference prints 5 digits here
    ours, want = run("testLMCubicLinearCoef")
    assert np.array_equal(vectors(ours)[-1], vectors(want)[-1])
    for driver in ("testGA", "testGAParallel"):                                  # same stream, same draws: bit for bit
        ours, want = run(driver)
        assert np.array_equal(vectors(ours, "at params:")[-1], vectors(want, "at params:")[-1]), driver
        assert scalar(ours, "At generation =") == scalar(want, "At generation =")
    for driver in ("testGradientEvaluation", "testGradientApproxMultMPIRecur"):
        ours, want = run(driver)
        a, b = vectors(ours), vectors(want)
        assert len(a) == len(b) and all(np.array_equal(u, v) for u, v in zip(a, b)), driver
