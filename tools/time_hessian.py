"""Analytic Hessian (pnol_hessian) against the forward difference (pnol_fd_hessian), in one process, the two alternated.

  1. one Hessian of Rosenbrock and Rastrigin at n = 10, 512 and 4096 (both paths), and the analytic path alone at n = 16384 and at the
     largest n that fits; the user's dense quadratic form (tests/user_functor/my_hessians.cu, built out of tree) at 4096 and 8192.
     CUDA events on the context's stream around a number of calls after a warm-up, with x, dx and H in device memory (no host staging
     is timed); best of ROUNDS alternated rounds. GB/s counts the algorithmic bytes: 8 n^2 written, plus 8 n^2 of A read for the
     quadratic form, against pnol_measure_copy_bandwidth (read + write bytes of a device-to-device copy) taken in the same run;
  2. hessian_kernel alone (torch.profiler, CUDA activities, after the timed calls of each row): the call of part 1 adds its launch
     and host synchronisation, about 0.012 ms (the n = 10 row);
  3. one Objective::hessianApproximation call through the plugin API with host vectors (hostapi.hessian) at n = 512 and 4096, in both
     modes of pnol::Runtime::setAnalyticHessian: wall time of the call, host copies included.

Prints the card and its power limit first; the numbers belong to them. Environment: ROUNDS (default 5), WINDOW_MS (default 50: the
calls per timed window are chosen to fill about this much GPU time)."""
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch  # noqa: E402

from parallelnonlinearoptimizationlibrary_b200 import capi, hostapi  # noqa: E402

ROUNDS = int(os.environ.get("ROUNDS", 5))
WINDOW_MS = float(os.environ.get("WINDOW_MS", 50))


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        return q.stdout.strip()
    except Exception as e:          # the numbers below then stand without their card: say so
        return "unknown (%s)" % e


def time_calls(stream, calls):
    """best ms per call of each callable, the callables alternated round by round"""
    reps = {}
    for mode, call in calls.items():
        for _ in range(3):
            assert call() == 0
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        assert call() == 0
        b.record(stream)
        b.synchronize()
        reps[mode] = int(min(500, max(3, WINDOW_MS / max(a.elapsed_time(b), 1e-3))))
    best = {m: float("inf") for m in calls}
    for _ in range(ROUNDS):
        for mode, call in calls.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            for _ in range(reps[mode]):
                call()
            b.record(stream)
            b.synchronize()
            best[mode] = min(best[mode], a.elapsed_time(b) / reps[mode])
    return best


def kernel_ms(call):
    """least device time of hessian_kernel over 10 calls (torch.profiler, CUDA activities); None when the trace has none"""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(10):
            call()
        torch.cuda.synchronize()
    us = [e.device_time for e in prof.events() if "hessian_kernel" in e.name and "fd_hessian" not in e.name]
    return min(us) / 1e3 if us else None


def main():
    print("card: %s" % card())
    ctx = capi.Context(0)
    stream = torch.cuda.ExternalStream(ctx.stream)
    lib = ctx.lib
    copy_gbs = ctx.measure_copy_bandwidth()
    nmax = (int(torch.cuda.get_device_properties(0).shared_memory_per_block_optin) - 32 * 33 * 8) // 8
    print("device-to-device copy: %.0f GB/s (read + write bytes); largest n of pnol_hessian: %d" % (copy_gbs, nmax))
    print("part 1: one Hessian, ms per call (best of %d rounds)" % ROUNDS)
    print("%-11s %6s %11s %11s %9s %9s %9s %11s %11s %9s %9s" % ("objective", "n", "fd", "analytic", "fd/anal.", "GB/s", "of copy",
                                                               "max|H diff|", "kernel", "GB/s", "of copy"))

    def row(name, f, n, with_fd, read_bytes=0):
        x = torch.from_numpy(np.random.default_rng(n).uniform(-2, 2, n)).cuda()
        dx = torch.full((n,), 1e-3, dtype=torch.float64, device="cuda")
        H = torch.empty((n, n), dtype=torch.float64, device="cuda")
        H2 = torch.empty((n, n), dtype=torch.float64, device="cuda") if with_fd else None
        torch.cuda.synchronize()
        calls = {"analytic": lambda: lib.pnol_hessian(ctx.h, f.handle, capi._ptr(x), n, capi._ptr(H))}
        if with_fd:
            calls["fd"] = lambda: lib.pnol_fd_hessian(ctx.h, f.handle, capi._ptr(x), capi._ptr(dx), n, capi._ptr(H2))
        best = time_calls(stream, calls)
        gbs = (8.0 * n * n + read_bytes) / (best["analytic"] * 1e-3) / 1e9
        fd = "%11.4f" % best["fd"] if with_fd else "%11s" % "-"
        ratio = "%9.1f" % (best["fd"] / best["analytic"]) if with_fd else "%9s" % "-"
        diff = "%11.3e" % float((H - H2).abs().max()) if with_fd else "%11s" % "-"
        km = kernel_ms(calls["analytic"])
        kgbs = (8.0 * n * n + read_bytes) / (km * 1e-3) / 1e9 if km else float("nan")
        print("%-11s %6d %s %11.4f %s %9.0f %9.2f %s %11.4f %9.0f %9.2f" % (name, n, fd, best["analytic"], ratio, gbs, gbs / copy_gbs, diff,
                                                                      km or float("nan"), kgbs, kgbs / copy_gbs), flush=True)
        del H, H2
        torch.cuda.empty_cache()

    for name, kind in (("rosenbrock", capi.F_ROSENBROCK), ("rastrigin", capi.F_RASTRIGIN)):
        f = ctx.functor(kind)
        for n in (10, 512, 4096):
            row(name, f, n, True)
        for n in (16384, nmax):
            row(name, f, n, False)
        f.close()
    import user_hessian_lib as UH
    UH.build_and_load()
    for n in (4096, 8192):
        A = torch.from_numpy(np.random.default_rng(n).normal(size=n * n)).cuda()
        f = ctx.functor(UH.MYH_F_QUADFORM, (), (), (A,), n * n)
        row("quadform", f, n, False, read_bytes=8.0 * n * n)
        f.close()
        del A

    print("part 3: Objective::hessianApproximation with host vectors (hostapi.hessian), ms per call (best of %d)" % ROUNDS)
    hostapi.attach(ctx)
    for n in (512, 4096):
        x = np.random.default_rng(n).uniform(-2, 2, n)
        dx = np.full(n, 1e-3)
        best = {}
        for _ in range(1 + ROUNDS):
            for mode in (False, True):
                hostapi.set_analytic_hessian(mode)
                t0 = time.perf_counter()
                hostapi.hessian("rosenbrock", x, dx)
                dt = (time.perf_counter() - t0) * 1e3
                key = "analytic" if mode else "fd"
                best[key] = min(best.get(key, float("inf")), dt)
        print("  rosenbrock n = %5d: fd %9.3f ms, analytic %9.3f ms" % (n, best["fd"], best["analytic"]))
    hostapi.set_analytic_hessian(False)
    hostapi.detach()
    ctx.close()


if __name__ == "__main__":
    main()
