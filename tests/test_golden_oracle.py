"""CPU: the oracle restatement (oracle/pnol_oracle.cpp) against the committed outputs of the VERBATIM reference
(tests/golden/ref_golden.npz, made by tests/golden/make_golden.py from /root/reference/Source + oracle/shim). Bit-exact."""
import os

import numpy as np
import pytest

import oracle_lib as O

G = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_golden.npz"))
KIND = {"rosenbrock": (1, ()), "booth": (3, ()), "goldstein": (4, ()), "powerprod3": (2, (3,)), "powerprod2": (2, (2,)), "rastrigin": (5, ())}


def g(case, name):
    return G["%s/%s" % (case, name)]


@pytest.mark.parametrize("spec,n", [("rosenbrock", 5), ("rosenbrock", 40), ("booth", 2), ("goldstein", 2), ("powerprod3", 5), ("rastrigin", 12)])
def test_fd_gradient_hessian(spec, n):
    case = "fdgrad_%s_%d" % (spec, n)
    kind, ints = KIND[spec]
    f = O.OFunctor(kind, (), ints)
    gr, f0 = O.fd_gradient(f, g(case, "x"), g(case, "dx"))
    assert np.array_equal(gr, g(case, "g")) and np.array_equal(gr, g(case, "g_mpi")) and f0 == g(case, "f")[0]
    if n <= 12:
        assert np.array_equal(O.fd_hessian(f, g(case, "x"), g(case, "dxh")), g(case, "B"))


def test_reference_known_answers():
    # SURVEY.md Appendix C; testGradientEvaluation (Source/Examples.cpp:512-540) uses libm pow(x,3): FD-noise level only
    assert g("testGradientEvaluation", "g")[0] == 27.000008998356861
    gr, _ = O.fd_gradient(O.OFunctor(2, (), (3,)), np.full(5, 3.0), np.full(5, 1e-6))
    assert np.allclose(gr, g("testGradientEvaluation", "g"), rtol=1e-7)
    assert np.allclose(g("testLMExpMPI", "X"), [10.2, 0.4, 0.1], rtol=1e-8)
    assert np.allclose(g("testLMCubicLinearCoef", "X"), [0.3, 1.1, -4.3, 7.3], rtol=1e-10)
    assert abs(g("testBFGS", "fOpt")[0] - 3.9308394359855199) < 1e-12


def test_recur():
    c = "recur_rosenbrock_8"
    gr, f0 = O.fd_gradient_recur(O.OFunctor(1), g(c, "xr"), np.full(7, 1e-6), g(c, "constx"), g(c, "ind"))
    assert np.array_equal(gr, g(c, "g")) and np.array_equal(gr, g(c, "g_mpi")) and f0 == g(c, "f")[0]


@pytest.mark.parametrize("K", [4, 32, 128])
def test_fd_jacobian(K):
    c = "fdjac_lorentz_K%d" % K
    t = g(c, "t")
    f = O.OFunctor(103, (float(g(c, "w")),), (), (t, g(c, "y")), t.size)
    J, F = O.fd_jacobian(f, g(c, "x"), g(c, "dx"))
    assert np.array_equal(J, g(c, "J")) and np.array_equal(J, g(c, "J_mpi")) and np.array_equal(F, g(c, "F"))


@pytest.mark.parametrize("K", [8, 16])
def test_lm(K):
    c = "lm_lorentz_K%d" % K
    t = g(c, "t")
    f = O.OFunctor(103, (float(g(c, "w")),), (), (t, g(c, "y")), t.size)
    w = O.lm(f, g(c, "x0"), 0.001, 10.0, 1e-7, int(g(c, "iters")), 0.0)
    assert np.array_equal(w["X"], g(c, "X")) and np.array_equal(w["F"], g(c, "F")) and np.array_equal(w["F0"], g(c, "F0"))


@pytest.mark.parametrize("n", [3, 17, 64])
def test_update_hinv(n):
    c = "updhinv_%d" % n
    assert np.array_equal(O.update_hinv(g(c, "D"), g(c, "g"), g(c, "s")), g(c, "Dnew"))


def test_box():
    assert O.compute_alpha_bnd(g("box", "xin"), g("box", "lb"), g("box", "ub"), g("box", "p")) == g("box", "alphabnd")[0]
    xw, cnt = O.check_box_bounds(g("box", "x"), g("box", "lb"), g("box", "ub"))
    assert cnt > 0 and np.array_equal(xw, g("box", "Xfixed"))


@pytest.mark.parametrize("spec", ["powerprod2", "rastrigin", "rosenbrock"])
def test_ga(spec):
    c = "ga_%s" % spec
    kind, ints = KIND[spec]
    w = O.ga(O.OFunctor(kind, (), ints), g(c, "x0"), g(c, "lb"), g(c, "ub"), int(g(c, "npop")), int(g(c, "gens")),
             dict(seed=int(g(c, "seed")), scale=float(g(c, "scale"))))
    assert np.array_equal(w["X"], g(c, "X")) and w["fOpt"] == g(c, "fOpt")[0] and w["f0"] == g(c, "f0")[0]
    assert w["stream_pos"] == int(g(c, "stream_pos")[0])


def test_ga_stages():
    c = "ga_stages"
    Xs, Fs = O.ga_pop_sort(g(c, "X"), g(c, "F"))
    assert np.array_equal(Xs, g(c, "sortedX")) and np.array_equal(Fs, g(c, "sortedF"))
    Xb, ib, pb = O.ga_check_bounds(g(c, "X"), g(c, "lb"), g(c, "ub"), dict(seed=5, scale=1.0))
    assert np.array_equal(Xb, g(c, "boundsX")) and np.array_equal(ib, g(c, "boundsInd")) and pb == int(g(c, "boundsPos")[0])
    Xi, ii, pi = O.ga_check_identical(g(c, "X"), g(c, "lb"), g(c, "ub"), dict(seed=5, scale=1.0))
    assert np.array_equal(Xi, g(c, "identX")) and np.array_equal(ii, g(c, "identInd")) and pi == int(g(c, "identPos")[0])


def test_simplex_golden_is_what_the_verbatim_reference_produces():
    # tests/golden/simplex_golden.npz: every case stored, the known answers of the reference's example drivers, and a fresh run
    # of the reference's SimplexSearch::findMin where oracle/_ref is built
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    sys.path.insert(0, os.path.join(here, "golden"))
    import make_simplex_golden as M
    G2 = np.load(os.path.join(here, "golden", "simplex_golden.npz"))
    for name in M.CASES:
        for k in ("X", "f0", "fOpt", "stream_pos"):
            assert name + "/" + k in G2.files, (name, k)
    # Rosenbrock -> 1, Booth -> (1, 3), Goldstein-Price -> (0, -1) with f = 3
    assert np.allclose(G2["rosenbrock4/X"], 1.0, atol=1e-6) and np.allclose(G2["booth/X"], [1.0, 3.0], atol=1e-6)
    assert np.allclose(G2["goldstein/X"], [0.0, -1.0], atol=1e-6) and abs(G2["goldstein/fOpt"][0] - 3.0) < 1e-9
    if O.have_ref():
        for name, (obj, x0, kw, stream) in M.CASES.items():
            r = M.run_reference(obj, x0, kw, stream)
            for k in ("X", "f0", "fOpt", "stream_pos"):
                assert np.array_equal(r[k], G2[name + "/" + k]), (name, k)


def test_bfgsbnd_mpi_golden_is_what_the_verbatim_reference_produces():
    # tests/golden/bfgsbnd_mpi_golden.npz against a fresh run of the reference's BFGSBnd_MPI::findMinBnd (needs oracle/_ref), and
    # the known answers of that driver: the bounded example ends on Xlb[0] = -1 at the n = 10 minimum f = 4 when the pool is wide
    # enough, and the serial-equivalent pool of 2 lands in the f = 3.9866 local minimum (SURVEY.md Appendix C)
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    sys.path.insert(0, os.path.join(here, "golden"))
    import make_bfgsbnd_mpi_golden as M
    G2 = np.load(os.path.join(here, "golden", "bfgsbnd_mpi_golden.npz"))
    cases = M.cases()
    assert sorted(set(k.split("/")[0] for k in G2.files)) == sorted(cases)
    for name, (obj, x0, lb, ub, P, iters, extra, twin) in cases.items():
        X = G2[name + "/X"]
        assert np.array_equal(G2[name + "/x0"], x0) and int(G2[name + "/P"]) == P and int(G2[name + "/iters"]) == iters
        assert np.all(X >= lb) and np.all(X <= ub) and G2[name + "/fOpt"][0] <= G2[name + "/f0"][0]
        assert ("X_ulp" in "".join(k for k in G2.files if k.startswith(name + "/"))) == twin
    for P in (4, 8):
        c = "example_P%d_it200" % P
        assert G2[c + "/X"][0] == -1.0 and abs(G2[c + "/fOpt"][0] - 4.0) < 1e-6 and int(G2[c + "/recursions"]) == 1
    assert abs(G2["example_P2_it200/fOpt"][0] - 3.98658) < 1e-5
    assert np.array_equal(G2["power2_allfrozen_P4/X"], np.full(5, 0.5)) and G2["power2_allfrozen_P4/fOpt"][0] == 1.25
    if O.have_ref():
        for name, (obj, x0, lb, ub, P, iters, extra, twin) in cases.items():
            r = M.run_reference(obj, x0, lb, ub, P, iters, extra)
            for k in ("X", "f0", "fOpt"):
                assert np.array_equal(r[k], G2[name + "/" + k]), (name, k)


def test_alpha_pool_oracle_against_the_committed_reference_outputs():
    # tests/golden/alphapool_golden.npz = BFGS_Bnd_MPI_SW::evaluateAlphaPoolAndDerivatives of the verbatim reference (4 ranks): the
    # oracle's phi / slope / sentinel bit for bit, with and without an active set; fresh-run comparison where oracle/_ref exists
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    sys.path.insert(0, os.path.join(here, "golden"))
    import make_alphapool_golden as M
    G2 = np.load(os.path.join(here, "golden", "alphapool_golden.npz"))
    for name, c in M.cases().items():
        assert np.array_equal(G2[name + "/x"], c["x"]) and np.array_equal(G2[name + "/p"], c["p"])
        f = O.OFunctor(c["kind"], (), c["ints"])
        phi, dphi, bad = O.alpha_pool(f, c["x"], c["p"], c["alpha"], c["dalpha"], const_x=c["constx"], const_ind=c["ind"])
        assert np.array_equal(phi, G2[name + "/phi"]), name
        assert np.array_equal(dphi, G2[name + "/dphi"], equal_nan=True), name
        assert bad == int(np.sum(G2[name + "/phi"] == 1e10))
        if O.have_ref():
            r = M.run_reference(c, nprocs=2)
            assert np.array_equal(r["phi"], G2[name + "/phi"]) and np.array_equal(r["dphi"], G2[name + "/dphi"], equal_nan=True)
    assert np.all(G2["rosenbrock6_overflow/phi"] == 1e10)


# ---- BASELINE.json shapes (tests/golden/baseline_lm_golden.npz, made by tests/golden/make_baseline_lm_golden.py) ----
GB = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "baseline_lm_golden.npz"))


@pytest.mark.parametrize("K,m,iters", [(8, 3000, 8), (32, 1500, 5), (128, 300, 3)])
def test_threaded_lm_restatement_equals_the_sequential_one(K, m, iters):
    # oracle_lm_mt (loops re-nested, rows / bands of J^T J dealt to threads) must give oracle_lm's bits at any thread count
    from parallelnonlinearoptimizationlibrary_b200 import problems
    pr = problems.lorentz_problem(m, K)
    f = O.OFunctor(103, (pr["w"],), (), (pr["t"], pr["y"]), m)
    a = O.lm(f, pr["x0"], 0.001, 10.0, 1e-7, iters, 0.0, want_trace=True)
    for threads in (1, 3, 8):
        b = O.lm_mt(f, pr["x0"], 0.001, 10.0, 1e-7, iters, 0.0, want_trace=True, threads=threads)
        assert a["iters"] == b["iters"] and a["chisq"] == b["chisq"] and a["lam"] == b["lam"]
        assert np.array_equal(a["X"], b["X"]) and np.array_equal(a["F"], b["F"]) and np.array_equal(a["F0"], b["F0"])
        assert np.array_equal(a["trace"], b["trace"], equal_nan=True)


@pytest.mark.parametrize("case", ["cfg2_it6", "cfg2_to_stop", "lm_K128"])
def test_baseline_shape_lm_golden_is_what_the_oracle_produces(case):
    # cfg2 at FULL size (m = 100k, n = 16) and n = 256 (K = 128): the committed outputs of the verbatim reference, bit for bit
    from parallelnonlinearoptimizationlibrary_b200 import problems
    q = lambda k: GB["%s/%s" % (case, k)]      # noqa: E731
    pr = problems.lorentz_problem(int(q("m")), int(q("K")))
    f = O.OFunctor(103, (pr["w"],), (), (pr["t"], pr["y"]), pr["m"])
    w = O.lm_mt(f, pr["x0"], float(q("lambda0")), float(q("factor")), float(q("dxgrad")), int(q("maxiter")), float(q("xmindiff")))
    assert w["iters"] == int(q("iters")) and np.array_equal(w["X"], q("X")) and w["chisq"] == float(q("chisq"))
    if case == "lm_K128":
        assert np.array_equal(w["F"], q("F")) and np.array_equal(w["F0"], q("F0"))
    else:
        assert np.array_equal(w["F"][::100], q("F_every100")) and np.array_equal(w["F0"][::100], q("F0_every100"))
