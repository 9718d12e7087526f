"""Batches of small fitting problems for the batched Levenberg-Marquardt tests (pnol_lm_batch, LevMarqBatch), and their references:
oracle_lib.lm on each problem alone (its columns sliced), and a Python restatement of the same loop over oracle_lib.lm_normal_eq /
lu_solve for models the oracle does not know and for the analytic Jacobian."""
import numpy as np

import oracle_lib as O
from parallelnonlinearoptimizationlibrary_b200 import capi

LORENTZ_W = 40.0


def model_data(kind, n, m, rng):
    """(scalars, columns, true x, start x) of one problem with m rows"""
    if kind == capi.F_EXPCURVE:
        t = np.linspace(0.0, 2.0, m)
        xt = np.array([rng.uniform(1, 3), rng.uniform(-1, 1), rng.uniform(-0.5, 0.5)])
        y = xt[0] * np.exp(xt[1] * t) + xt[2] + 1e-3 * rng.standard_normal(m)
        return (), (t, y), xt, xt * rng.uniform(0.8, 1.2, 3)
    if kind == capi.F_CUBIC:
        x = np.linspace(-2.0, 2.0, m)
        xt = rng.uniform(-2, 2, 4)
        y = xt[0] * x ** 3 + xt[1] * x * x + xt[2] * x + xt[3] + 1e-3 * rng.standard_normal(m)
        return (), (x ** 3, x, y), xt, xt + rng.uniform(-0.5, 0.5, 4)
    # sum of Lorentzians (built-in, or the user copy of tests/user_functor/my_jacobians.hpp), and the user Gaussian peak
    if kind == 2102:
        t = np.linspace(-2.0, 2.0, m)
        xt = np.array([rng.uniform(1, 2), rng.uniform(-0.5, 0.5), rng.uniform(0.5, 2)])
        y = xt[0] * np.exp(-(t - xt[1]) ** 2 * xt[2]) + 0.1 + 1e-3 * rng.standard_normal(m)
        return (0.1,), (t, y), xt, xt * rng.uniform(0.9, 1.1, 3)
    K = n // 2
    t = np.linspace(-0.5, 1.5, m)
    a = rng.uniform(1, 2, K)
    c = (np.arange(K) + rng.uniform(0.3, 0.7, K)) / K
    xt = np.empty(n)
    xt[0::2], xt[1::2] = a, c
    y = np.zeros(m)
    for k in range(K):
        y += a[k] / (1 + LORENTZ_W * (t - c[k]) ** 2)
    y += 1e-3 * rng.standard_normal(m)
    x0 = xt.copy()
    x0[0::2] *= rng.uniform(0.9, 1.1, K)
    x0[1::2] += rng.uniform(-0.02, 0.02, K) / K
    return (LORENTZ_W,), (t, y), xt, x0


def make_batch(kind, n, sizes, seed=0):
    """B = len(sizes) problems of the model, back to back: dict(kind, n, scalars, columns, row_off, X0, Xtrue)"""
    rng = np.random.default_rng(seed)
    cols, X0, Xt = None, [], []
    scalars = ()
    for m in sizes:
        scalars, c, xt, x0 = model_data(kind, n, int(m), rng)
        cols = [list(cc) for cc in c] if cols is None else [a + list(cc) for a, cc in zip(cols, c)]
        X0.append(x0)
        Xt.append(xt)
    row_off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    return dict(kind=kind, n=n, scalars=scalars, columns=[np.array(c, dtype=np.float64) for c in cols], row_off=row_off,
                X0=np.array(X0, dtype=np.float64).reshape(len(sizes), n), Xtrue=np.array(Xt).reshape(len(sizes), n))


def problem_columns(case, b):
    lo, hi = case["row_off"][b], case["row_off"][b + 1]
    return [np.ascontiguousarray(c[lo:hi]) for c in case["columns"]], int(hi - lo)


def oracle_problem(case, b, lambda0, factor, dxgrad, maxiter, xmindiff, kind=None):
    """oracle_lm on problem b alone: dict(X, F, iters, chisq, lam, stopped)"""
    cols, m = problem_columns(case, b)
    of = O.OFunctor(case["kind"] if kind is None else kind, case["scalars"], (), cols, m)
    r = O.lm(of, case["X0"][b], lambda0, factor, dxgrad, maxiter, xmindiff)
    r["stopped"] = int(r["iters"] < maxiter)
    return r


def _sumsq(F):
    return float(np.cumsum(F * F)[-1]) if F.size else 0.0       # s = s + F_k F_k, k ascending (cumsum is a running sum)


def py_lm(resid, jac, x0, lambda0, factor, maxiter, xmindiff):
    """oracle_lm's loop (Source/LevenbergMarquardtMPI.cpp:12-173) in Python over oracle_lib's normal equations and LU solve.
    resid(x) -> F, jac(x, F) -> J (m x n)"""
    X = np.array(x0, dtype=np.float64)
    lam = lambda0
    F = resid(X)
    chi = np.sqrt(_sumsq(F)) ** 2
    it, stopped = 0, 0
    while it < maxiter:
        J = jac(X, F)
        _, A, rhs = O.lm_normal_eq(J.reshape(F.size, X.size), F, lam)
        sig = O.lu_solve(A, rhs)
        Xt = X + sig
        Ft = resid(Xt)
        ct = np.sqrt(_sumsq(Ft)) ** 2
        if ct >= chi or ct != ct:
            lam = lam * factor
        else:
            lam = lam / factor
            chi, X, F = ct, Xt, Ft
            if np.sqrt(_sumsq(sig)) < xmindiff:
                stopped = 1
                break
        it += 1
    return dict(X=X, F=F, iters=it, chisq=chi, lam=lam, stopped=stopped)


def fd_jac(resid, dx):
    """the forward-difference Jacobian of oracle_fd_jacobian: (r(X + dx e_j) - r(X)) / dx"""
    def jac(X, F):
        J = np.empty((F.size, X.size))
        for j in range(X.size):
            Xp = X.copy()
            Xp[j] = Xp[j] + dx
            J[:, j] = (resid(Xp) - F) / dx
        return J
    return jac
