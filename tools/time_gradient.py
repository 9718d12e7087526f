"""Analytic gradient (pnol_gradient) against the forward difference (pnol_fd_gradient), in one process, the two alternated.

  1. one gradient of Rosenbrock and Rastrigin at n = 10, 512 and 4096: CUDA events on the context's stream around REPS calls after a
     warm-up, with x, dx and g in device memory (so no host staging is timed); best of ROUNDS alternated rounds;
  2. cfg3 end to end: BFGS_Bnd_MPI_SW on Rosenbrock at n = 4096 with pool width 8 and 20 iterations (tools/time_bfgs.py's start point),
     in both modes of pnol::Runtime::setAnalyticGradient: wall time per iteration and the final f.

Prints the card and its power limit first; the numbers belong to them. Environment: REPS (default 200), ROUNDS (default 5)."""
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


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        return q.stdout.strip()
    except Exception as e:          # the numbers below then stand without their card: say so
        return "unknown (%s)" % e


def main():
    print("card: %s" % card())
    ctx = capi.Context(0)
    stream = torch.cuda.ExternalStream(ctx.stream)
    lib = ctx.lib
    print("part 1: one gradient, ms per call (best of %d rounds of %d calls)" % (ROUNDS, REPS))
    print("%-11s %6s %10s %10s %8s %12s" % ("objective", "n", "fd", "analytic", "ratio", "max|g diff|"))
    for name, kind in (("rosenbrock", capi.F_ROSENBROCK), ("rastrigin", capi.F_RASTRIGIN)):
        f = ctx.functor(kind)
        for n in (10, 512, 4096):
            x = torch.from_numpy(np.random.default_rng(n).uniform(-2, 2, n)).cuda()
            dx = torch.full((n,), 1e-7, dtype=torch.float64, device="cuda")
            g = torch.empty(n, dtype=torch.float64, device="cuda")
            torch.cuda.synchronize()
            calls = {
                "fd": lambda: lib.pnol_fd_gradient(ctx.h, f.handle, capi._ptr(x), capi._ptr(dx), n, capi._ptr(g), None),
                "analytic": lambda: lib.pnol_gradient(ctx.h, f.handle, capi._ptr(x), n, capi._ptr(g), None),
            }
            out = {}
            for mode, call in calls.items():
                for _ in range(20):
                    assert call() == 0, lib.pnol_last_error(ctx.h)
                out[mode] = g.cpu().numpy().copy()
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
            diff = float(np.max(np.abs(out["fd"] - out["analytic"])))
            print("%-11s %6d %10.4f %10.4f %8.2f %12.3e" % (name, n, best["fd"], best["analytic"], best["fd"] / best["analytic"], diff))
        f.close()

    print("part 2: cfg3, BFGS_Bnd_MPI_SW on Rosenbrock, n = 4096, pool width 8, 20 iterations")
    hostapi.attach(ctx)
    n = 4096
    SW = [1e-4, 0.8, 1e-6, 1.0, 1e-10, 2.0, 50, 1e-5, 1e-6, 1e-3, 20, 1e-5, 1e-5, 0]
    x0 = np.full(n, 2.0)
    x0[0] = -5.0
    lb, ub = np.full(n, -5.0), np.full(n, 5.0)
    res = {}
    for rnd in range(1 + ROUNDS // 2):
        for mode in (False, True):
            hostapi.set_analytic_gradient(mode)
            if rnd == 0:           # warm-up
                hostapi.bfgs("bfgs_bnd_sw", "rosenbrock", x0, SW[:10] + [2] + SW[11:], lb, ub, pool_width=8)
            ctx.sync()
            t0 = time.perf_counter()
            r = hostapi.bfgs("bfgs_bnd_sw", "rosenbrock", x0, SW, lb, ub, pool_width=8)
            ctx.sync()
            dt = (time.perf_counter() - t0) / r["iterations"] * 1e3
            key = "analytic" if mode else "fd"
            if key not in res or dt < res[key][0]:
                res[key] = (dt, r["fOpt"], r["iterations"])
    hostapi.set_analytic_gradient(False)
    for key in ("fd", "analytic"):
        dt, fo, it = res[key]
        print("  %-9s %8.3f ms per iteration (best of %d), %d iterations, final f = %.17g" % (key, dt, 1 + ROUNDS // 2, it, fo))
    hostapi.detach()
    ctx.close()


if __name__ == "__main__":
    main()
