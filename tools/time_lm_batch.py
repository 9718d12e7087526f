"""Timing of the batched Levenberg-Marquardt (pnol_lm_batch, DESIGN.md section 4.5).

Shapes: the sum of Lorentzians with K = 2 (n = 4, 256 rows a problem) and K = 8 (n = 16, 1024 rows a problem), B = 65 536 problems,
50 iterations each (x_min_diff = 0: no problem stops early), the forward-difference and the analytic Jacobian alternated in one process,
timed with CUDA events. Reported per shape and mode: the batch time, fits/s, problem-iterations/s (counted from the iterations the
kernel reports), and an FP64 operation count of the algorithm from the shapes (the model's FP64 operations per residual row as stated
below, times the rows it evaluates, plus the sums) over the time. For comparison, labelled as estimates: the same problems through one
pnol_lm_iterate loop per problem (a sample of 64 problems timed, extrapolated to B), and the oracle (oracle_lib.lm, one problem per host
core: a sample timed on one core, extrapolated to B over os.cpu_count() cores).

    python tools/time_lm_batch.py [--B 65536] [--iters 50] [--reps 3] [--out results.json]

Every shape is printed as JSON; --out also writes the whole result to that file.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

W = 40.0
# FP64 operations of one sum-of-Lorentzians residual row per term: t - c, d*d, w*q, 1 + e, a / den (a division: about 8 FP64
# operations on the device) and one tree addition; plus y - S. Analytic Jacobian row per term: the same four, 1/den, and five more.
OPS_TERM_RESID = 4 + 8 + 1
OPS_TERM_JAC = 4 + 8 + 5


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return q.stdout.strip()
    except Exception as e:       # the numbers are still worth having; say that the card could not be read
        return "nvidia-smi unavailable: %s" % e


def lorentz_batch(B, K, mb, seed):
    rng = np.random.default_rng(seed)
    t1 = np.linspace(-0.5, 1.5, mb)
    a = rng.uniform(1, 2, (B, K))
    c = (np.arange(K) + rng.uniform(0.3, 0.7, (B, K))) / K
    y = np.zeros((B, mb))
    for k in range(K):
        y += a[:, k:k + 1] / (1 + W * (t1[None, :] - c[:, k:k + 1]) ** 2)
    y += 1e-3 * rng.standard_normal((B, mb))
    X0 = np.empty((B, 2 * K))
    X0[:, 0::2] = a * rng.uniform(0.9, 1.1, (B, K))
    X0[:, 1::2] = c + rng.uniform(-0.02, 0.02, (B, K)) / K
    return np.tile(t1, B), y.ravel(), X0


def op_count(K, mb, iters, jpasses, analytic):
    """FP64 operations of the batch (one problem): the model's rows plus the sums (see the module docstring)"""
    n = 2 * K
    resid = K * OPS_TERM_RESID + 1
    jrow = (K * OPS_TERM_JAC + resid) if analytic else ((n + 1) * resid + 2 * n)
    nsums = n * (n + 1) // 2 + n
    per_jpass = mb * (jrow + 2 * nsums)
    per_iter = mb * (resid + 2) + n ** 3 // 3 * 2        # the trial residuals and their squares, the LU
    return jpasses * per_jpass + iters * per_iter + mb * (resid + 2)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=65536)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--loop-sample", type=int, default=64)
    ap.add_argument("--oracle-sample", type=int, default=4)
    ap.add_argument("--out", default=None, help="also write the result as JSON to this file")
    a = ap.parse_args()
    import torch
    import oracle_lib as O
    from parallelnonlinearoptimizationlibrary_b200 import capi

    ctx = capi.Context(0)
    dev = torch.device("cuda:0")
    res = dict(gpu=gpu_info(), B=a.B, iters=a.iters, shapes=[])
    for K, mb in ((2, 256), (8, 1024)):
        n = 2 * K
        t, y, X0 = lorentz_batch(a.B, K, mb, seed=K)
        f = ctx.functor(capi.F_LORENTZ_SUM, (W,), (), (t, y), t.size)
        ro = torch.tensor(np.arange(a.B + 1, dtype=np.int64) * mb, device=dev)
        dx = torch.full((n,), 1e-7, dtype=torch.float64, device=dev)
        X0d = torch.tensor(X0, device=dev)
        Xd = torch.empty_like(X0d)
        outs = dict(chisq=torch.empty(a.B, dtype=torch.float64, device=dev), lam=torch.empty(a.B, dtype=torch.float64, device=dev),
                    iters=torch.empty(a.B, dtype=torch.int32, device=dev), stopped=torch.empty(a.B, dtype=torch.int32, device=dev))
        times = {capi.JAC_AUTO: [], capi.JAC_ANALYTIC: []}
        for rep in range(a.reps + 1):                          # rep 0 warms both modes up
            for mode in (capi.JAC_AUTO, capi.JAC_ANALYTIC):
                Xd.copy_(X0d)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                e0.record()
                ctx.lm_batch(f, ro, Xd, dx, 1e-3, 10.0, 0.0, a.iters, mode, n=n, B=a.B, out=outs)
                e1.record()
                torch.cuda.synchronize()
                if rep:
                    times[mode].append(e0.elapsed_time(e1) * 1e-3)
        shape = dict(K=K, n=n, rows=mb, modes={})
        for mode, name in ((capi.JAC_AUTO, "fd"), (capi.JAC_ANALYTIC, "analytic")):
            Xd.copy_(X0d)
            ctx.lm_batch(f, ro, Xd, dx, 1e-3, 10.0, 0.0, a.iters, mode, n=n, B=a.B, out=outs)
            it = int(outs["iters"].sum().item())
            tsec = float(np.median(times[mode]))
            ops = op_count(K, mb, a.iters, a.iters, mode == capi.JAC_ANALYTIC) * a.B     # upper bound: J recomputed every pass
            shape["modes"][name] = dict(seconds=tsec, all_times=times[mode], fits_per_s=a.B / tsec, problem_iters_per_s=it / tsec,
                                        fp64_ops_upper=ops, fp64_ops_per_s_upper=ops / tsec)
        # the per-problem loop: pnol_lm_iterate on one problem at a time (a sample, extrapolated)
        S = min(a.loop_sample, a.B)
        J = torch.empty(mb * n, dtype=torch.float64, device=dev)
        Fd = torch.empty(mb, dtype=torch.float64, device=dev)
        Ft = torch.empty(mb, dtype=torch.float64, device=dev)
        JTJ = torch.empty(n * n + n, dtype=torch.float64, device=dev)
        fs = []
        for b in range(S):
            fs.append(ctx.functor(capi.F_LORENTZ_SUM, (W,), (), (t[b * mb:(b + 1) * mb].copy(), y[b * mb:(b + 1) * mb].copy()), mb))
        dxh = np.full(n, 1e-7)

        def loop_one(fb, x0):
            F, ss = ctx.residual_eval(fb, x0, F=Fd, n=n)
            chi = np.sqrt(ss) ** 2
            ctx.lm_iterate(fb, x0, dxh, n, J, Fd, Ft, JTJ, 1e-3, chi, 10.0, a.iters, 0.0, capi.JAC_AUTO)

        loop_one(fs[0], X0[0])
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for b in range(S):
            loop_one(fs[b], X0[b])
        torch.cuda.synchronize()
        per = (time.perf_counter() - t0) / S
        shape["lm_iterate_loop_estimate"] = dict(sample=S, seconds_per_problem=per, seconds_for_B_extrapolated=per * a.B)
        for fb in fs:
            fb.close()
        # the oracle on the host cores (a sample on one core, extrapolated over all cores)
        So = a.oracle_sample
        t0 = time.perf_counter()
        for b in range(So):
            of = O.OFunctor(capi.F_LORENTZ_SUM, (W,), (), (t[b * mb:(b + 1) * mb], y[b * mb:(b + 1) * mb]), mb)
            O.lm(of, X0[b], 1e-3, 10.0, 1e-7, a.iters, 0.0)
        per = (time.perf_counter() - t0) / So
        cores = os.cpu_count() or 1
        shape["oracle_host_estimate"] = dict(sample=So, seconds_per_problem_one_core=per, cores=cores,
                                             seconds_for_B_extrapolated=per * a.B / cores)
        f.close()
        res["shapes"].append(shape)
        print(json.dumps(shape, indent=1), flush=True)
    ctx.close()
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)
    print(res["gpu"])


if __name__ == "__main__":
    main()
