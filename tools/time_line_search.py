"""Analytic line-search slopes (pnol_alpha_pool_analytic) against the forward-difference pool (pnol_alpha_pool), in one process.

  1. one pool call, pool width 8 (9 entries), Rosenbrock and Rastrigin at n = 10, 512 and 4096, x, p, alpha, phi and dphi in device
     memory: call time from CUDA events on the context's stream around REPS calls, each ending in the call's own synchronisation; best
     of ROUNDS rounds, the two calls alternated;
  2. kernel time of the same calls from torch.profiler, in a run of its own (this script started again with --profile): the pool
     kernel and its finish kernel, averaged over the profiled calls;
  3. cfg3 end to end: BFGS_Bnd_MPI_SW on Rosenbrock at n = 4096, pool width 8, 20 iterations (tools/time_bfgs.py's start point), with
     analytic gradients, with and without analytic slopes: wall time per iteration (best of the rounds), line-search iterations (pool
     calls, from the library's timers in a separate untimed run), objective evaluations and the final f;
  4. convergence: BFGS_Bnd_MPI_SW on Rosenbrock at n = 10 from x = 3 to minGrad2Norm = 1e-10 with analytic gradients, with
     forward-difference and with analytic slopes: iterations and whether the gradient stop was reached.

Prints the card and its power limit first; the numbers belong to them. Environment: REPS (default 200), ROUNDS (default 5)."""
import ctypes as C
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from parallelnonlinearoptimizationlibrary_b200 import capi, hostapi  # noqa: E402

REPS = int(os.environ.get("REPS", 200))
ROUNDS = int(os.environ.get("ROUNDS", 5))
NPOOL = 9
DALPHA = 1e-6
OBJECTIVES = (("rosenbrock", capi.F_ROSENBROCK), ("rastrigin", capi.F_RASTRIGIN))
SIZES = (10, 512, 4096)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        return q.stdout.strip()
    except Exception as e:          # the numbers below then stand without their card: say so
        return "unknown (%s)" % e


def pool_calls(ctx, f, n):
    """the two pool calls on device-resident data, and their outputs"""
    rng = np.random.default_rng(n)
    x = torch.from_numpy(rng.uniform(-2, 2, n)).cuda()
    p = torch.from_numpy(rng.normal(size=n) * 0.1).cuda()
    alpha = torch.from_numpy(np.linspace(0.0, 1.0, NPOOL)).cuda()
    out = {m: (torch.empty(NPOOL, dtype=torch.float64, device="cuda"), torch.empty(NPOOL, dtype=torch.float64, device="cuda")) for m in ("fd", "analytic")}
    lib, P = ctx.lib, capi._ptr
    torch.cuda.synchronize()
    calls = {
        "fd": lambda: lib.pnol_alpha_pool(ctx.h, f.handle, P(x), P(p), n, P(alpha), NPOOL, C.c_double(DALPHA), None, None, None, n,
                                          P(out["fd"][0]), P(out["fd"][1]), None),
        "analytic": lambda: lib.pnol_alpha_pool_analytic(ctx.h, f.handle, P(x), P(p), n, P(alpha), NPOOL, None, None, None, n,
                                                         P(out["analytic"][0]), P(out["analytic"][1]), None),
    }
    return calls, out


def part1(ctx):
    stream = torch.cuda.ExternalStream(ctx.stream)
    print("part 1: one pool call (%d entries), ms per call including its synchronisation (best of %d rounds of %d calls)" % (NPOOL, ROUNDS, REPS))
    print("%-11s %6s %10s %10s %8s %10s %14s" % ("objective", "n", "fd", "analytic", "ratio", "phi same", "max|dphi diff|"))
    for name, kind in OBJECTIVES:
        f = ctx.functor(kind)
        for n in SIZES:
            calls, out = pool_calls(ctx, f, n)
            for call in calls.values():
                for _ in range(20):
                    assert call() == 0, ctx.lib.pnol_last_error(ctx.h)
            best = {m: float("inf") for m in calls}
            for _ in range(ROUNDS):
                for mode, call in calls.items():
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record(stream)
                    for _ in range(REPS):
                        call()
                    b.record(stream)
                    b.synchronize()
                    best[mode] = min(best[mode], a.elapsed_time(b) / REPS)
            same = torch.equal(out["fd"][0], out["analytic"][0])
            diff = float((out["fd"][1] - out["analytic"][1]).abs().max())
            print("%-11s %6d %10.4f %10.4f %8.2f %10s %14.3e" % (name, n, best["fd"], best["analytic"], best["fd"] / best["analytic"], same, diff))
        f.close()


def profile(ctx):
    """kernel times of the pool calls (run with --profile, a process of its own)"""
    from torch.profiler import ProfilerActivity, profile as tprofile
    print("part 2: kernel time per call from torch.profiler, us (pool kernel + finish kernel), %d calls each" % REPS)
    print("%-11s %6s %-9s %12s %12s" % ("objective", "n", "mode", "pool kernel", "finish"))
    for name, kind in OBJECTIVES:
        f = ctx.functor(kind)
        for n in SIZES:
            calls, _ = pool_calls(ctx, f, n)
            for mode, call in calls.items():
                for _ in range(20):
                    call()
                torch.cuda.synchronize()
                with tprofile(activities=[ProfilerActivity.CUDA]) as prof:
                    for _ in range(REPS):
                        call()
                    torch.cuda.synchronize()
                pool_us, fin_us = 0.0, 0.0
                for ev in prof.key_averages():
                    t = getattr(ev, "device_time_total", None)
                    if t is None:
                        t = ev.cuda_time_total
                    if "alpha_pool_kernel" in ev.key or "alpha_slope_kernel" in ev.key:
                        pool_us += t / REPS
                    elif "finish_kernel" in ev.key:
                        fin_us += t / REPS
                print("%-11s %6d %-9s %12.2f %12.2f" % (name, n, mode, pool_us, fin_us))
        f.close()


def part3(ctx):
    print("part 3: cfg3, BFGS_Bnd_MPI_SW on Rosenbrock, n = 4096, pool width 8, 20 iterations, analytic gradients")
    hl = hostapi.lib()
    hl.pnolhost_last_evaluations.restype = C.c_longlong
    hostapi.attach(ctx)
    hostapi.set_analytic_gradient(True)
    n = 4096
    SW = [1e-4, 0.8, DALPHA, 1.0, 1e-10, 2.0, 50, 1e-5, 1e-6, 1e-3, 20, 1e-5, 1e-5, 0]
    x0 = np.full(n, 2.0)
    x0[0] = -5.0
    lb, ub = np.full(n, -5.0), np.full(n, 5.0)
    res = {}
    modes = (("fd slopes", False), ("analytic slopes", True))
    for rnd in range(1 + ROUNDS // 2):
        for key, mode in modes:
            hostapi.set_analytic_slope(mode)
            if rnd == 0:           # warm-up
                hostapi.bfgs("bfgs_bnd_sw", "rosenbrock", x0, SW[:10] + [2] + SW[11:], lb, ub, pool_width=8)
            ctx.sync()
            t0 = time.perf_counter()
            r = hostapi.bfgs("bfgs_bnd_sw", "rosenbrock", x0, SW, lb, ub, pool_width=8)
            ctx.sync()
            dt = (time.perf_counter() - t0) / r["iterations"] * 1e3
            if key not in res or dt < res[key][0]:
                res[key] = (dt, r["fOpt"], r["iterations"], hl.pnolhost_last_evaluations())
    for key, mode in modes:
        hostapi.set_analytic_slope(mode)
        ctx.timer_enable(True)
        ctx.timer_reset()
        hostapi.bfgs("bfgs_bnd_sw", "rosenbrock", x0, SW, lb, ub, pool_width=8)
        pools = ctx.timer_get("alpha_slope" if mode else "alpha_pool")[1]
        ctx.timer_enable(False)
        dt, fo, it, ev = res[key]
        print("  %-16s %8.3f ms per iteration (best of %d), %d iterations, %d line-search iterations (pool calls), %d objective "
              "evaluations, final f = %.17g" % (key, dt, 1 + ROUNDS // 2, it, pools, ev, fo))
    hostapi.set_analytic_slope(False)
    hostapi.set_analytic_gradient(False)
    hostapi.detach()


def part4(ctx):
    print("part 4: convergence, BFGS_Bnd_MPI_SW on Rosenbrock, n = 10 from x = 3, minGrad2Norm = 1e-10, analytic gradients")
    hostapi.attach(ctx)
    hostapi.set_analytic_gradient(True)
    n, tol, maxit = 10, 1e-10, 2000
    SW = [1e-4, 0.8, DALPHA, 1.0, 1e-10, 2.0, 50, 1e-5, 1e-6, 1e-3, maxit, 1e-300, tol, 0]   # xMinDiff: no step-size stop
    lb, ub = np.full(n, -5.0), np.full(n, 5.0)
    f = ctx.functor(capi.F_ROSENBROCK)
    for key, mode in (("fd slopes", False), ("analytic slopes", True)):
        hostapi.set_analytic_slope(mode)
        r = hostapi.bfgs("bfgs_bnd_sw", "rosenbrock", np.full(n, 3.0), SW, lb, ub, pool_width=8)
        g = np.linalg.norm(ctx.gradient(f, r["X"])[0])
        print("  %-16s %5d iterations, |g| = %.3e, gradient stop %s, |x - 1| = %.3e, f = %.6e"
              % (key, r["iterations"], g, "reached" if g < tol else "not reached", np.linalg.norm(r["X"] - 1.0), r["fOpt"]))
    f.close()
    hostapi.set_analytic_slope(False)
    hostapi.set_analytic_gradient(False)
    hostapi.detach()


def main():
    ctx = capi.Context(0)
    if "--profile" in sys.argv:
        profile(ctx)
        ctx.close()
        return
    print("card: %s" % card())
    part1(ctx)
    sys.stdout.flush()
    subprocess.run([sys.executable, os.path.abspath(__file__), "--profile"], check=True)
    part3(ctx)
    part4(ctx)
    ctx.close()


if __name__ == "__main__":
    main()
