"""Times the Jacobian + residual kernels at the cfg5 shape (CUDA-event scopes inside the library). Tuning helper.

PROF_JAC=fd (default) | analytic | both: the forward-difference Jacobian (PNOL_JAC_AUTO) and / or the analytic one
(PNOL_JAC_ANALYTIC), alternated in one process with `both`. Besides pnol_fd_jacobian alone, the "fd_jacobian" scope of pnol_lm_step is
timed: J + J^T F as an LM iteration pays for it, against the HBM roofline of its bytes (J written, t / y / F read) at the copy bandwidth
pnol_measure_copy_bandwidth measures in the same run.
PROF_USER=1: instead, the user's copy of the model (tests/user_functor/my_jacobians.cu, a registered functor) through the generic
analytic template against fd_jacobian_blackbox_kernel (n + 1 model evaluations per row), at PROF_M rows (default 1M)."""
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from parallelnonlinearoptimizationlibrary_b200 import capi, problems  # noqa: E402


def gpu_name():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                              timeout=30).stdout.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError, IndexError):
        return "unknown"


user = os.environ.get("PROF_USER", "0") == "1"
m = int(os.environ.get("PROF_M", 1_000_000 if user else 4_000_000))
K = int(os.environ.get("PROF_K", 128))
which = os.environ.get("PROF_JAC", "fd")
modes = {"fd": [capi.JAC_AUTO], "analytic": [capi.JAC_ANALYTIC], "both": [capi.JAC_AUTO, capi.JAC_ANALYTIC]}[which]
ctx = capi.Context(0)
bw = ctx.measure_copy_bandwidth()
print("gpu: %s; copy bandwidth %.1f GB/s" % (gpu_name(), bw))
pr = problems.lorentz_problem(m, K)
n = pr["n"]
kind = capi.F_LORENTZ_SUM
if user:
    import user_jacobian_lib as UJ
    UJ.build_and_load()
    kind = UJ.MYJ_F_LORENTZ
    modes = [capi.JAC_BLACKBOX, capi.JAC_ANALYTIC]
f = ctx.functor(kind, (pr["w"],), (), (pr["t"], pr["y"]), m)
Jd, Fd, Ftd, JTJd = ctx.malloc(m * n * 8), ctx.malloc(m * 8), ctx.malloc(m * 8), ctx.malloc((n * n + n) * 8)
xd, dxd = ctx.to_device(pr["x0"]), ctx.to_device(np.full(n, float(os.environ.get("PROF_DX", 1e-7))))
ctx.residual_eval(f, xd, F=Fd, n=n)
names = {capi.JAC_AUTO: "fd", capi.JAC_BLACKBOX: "blackbox", capi.JAC_ANALYTIC: "analytic"}


def timed(fn, reps, scope="fd_jacobian"):
    for _ in range(2):
        fn()
    ctx.timer_enable(True)
    ctx.timer_reset()
    for _ in range(reps):
        fn()
    ctx.sync()
    ms, c = ctx.timer_get(scope)
    ctx.timer_enable(False)
    return ms / c


res = {md: {"jac": [], "step": []} for md in modes}
for _ in range(3):                                               # alternated rounds
    for md in modes:
        res[md]["jac"].append(timed(lambda: ctx.fd_jacobian(f, xd, dxd, J=Jd, F=Fd, mode=md, n=n), 2 if user and md == capi.JAC_BLACKBOX else 10))
        if not user:
            res[md]["step"].append(timed(lambda: ctx.lm_step(f, xd, dxd, n, Jd, Fd, Ftd, 1e-3, JTJd, jac_mode=md), 10))
r = timed(lambda: ctx.residual_eval(f, xd, F=Fd, n=n), 10, "residual")
step_bytes = m * n * 8 + 3 * m * 8                               # J written; t, y, F read
for md in modes:
    j = min(res[md]["jac"])
    line = "%s m=%d n=%d kind=%d: pnol_fd_jacobian (J + F) %.4f ms (runs %s)" % (
        names[md], m, n, kind, j, " ".join("%.4f" % v for v in res[md]["jac"]))
    if not user:
        s = min(res[md]["step"])
        gbs = step_bytes / (s * 1e-3) / 1e9
        line += "; in pnol_lm_step (J + J^T F) %.4f ms = %.0f GB/s, %.2f of the copy bandwidth (runs %s)" % (
            s, gbs, gbs / bw, " ".join("%.4f" % v for v in res[md]["step"]))
    print(line)
print("residual %.4f ms" % r)
