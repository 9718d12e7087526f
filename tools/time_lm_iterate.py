"""Times the device-resident LM loop (pnol_lm_iterate, 10 iterations per call) at one rank's shape: per-iteration time with the
library's timer scopes off and on, and the sum of the scopes. PROF_M = 500000 is one rank's share of cfg5 at 8 GPUs. Tuning helper.
PROF_JAC=fd (default) | analytic | both: forward-difference (PNOL_JAC_AUTO) or analytic (PNOL_JAC_ANALYTIC) Jacobians; `both`
alternates the two in this process, three rounds each."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from parallelnonlinearoptimizationlibrary_b200 import capi, problems  # noqa: E402

K = int(os.environ.get("PROF_K", 128))
which = os.environ.get("PROF_JAC", "fd")
modes = {"fd": [("fd", capi.JAC_AUTO)], "analytic": [("analytic", capi.JAC_ANALYTIC)],
         "both": [("fd", capi.JAC_AUTO), ("analytic", capi.JAC_ANALYTIC)] * 3}[which]
ctx = capi.Context(0)
stream = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", 0))
for m in [int(v) for v in os.environ.get("PROF_M", "500000,4000000").split(",")]:
    pr = problems.lorentz_problem(m, K)
    n = pr["n"]
    f = ctx.functor(capi.F_LORENTZ_SUM, (pr["w"],), (), (pr["t"], pr["y"]), m)
    Jd, Fd, Ft, JTJd = ctx.malloc(m * n * 8), ctx.malloc(m * 8), ctx.malloc(m * 8), ctx.malloc((n * n + n) * 8)
    dx = np.full(n, 1e-7)

    def run(calls, jac_mode):
        X = None
        for _ in range(calls):
            _, ss = ctx.residual_eval(f, pr["x0"], F=Fd, n=n)
            X, lam, chi, acc, rej, _ = ctx.lm_iterate(f, pr["x0"].copy(), dx, n, Jd, Fd, Ft, JTJd, 1e-3, float(np.sqrt(ss) ** 2), 10.0, 10,
                                                      jac_mode=jac_mode)
        return X, lam, chi, acc, rej

    for name, jac_mode in modes:
        run(1, jac_mode)
        res = {}
        for timers in (False, True, False):
            ctx.timer_enable(timers)
            ctx.timer_reset()
            ctx.sync()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            out = run(4, jac_mode)
            e1.record(stream)
            ctx.sync()
            torch.cuda.synchronize()
            res[timers] = e0.elapsed_time(e1) / 40
            if timers:
                scopes = {}
                for k in ("fd_jacobian", "syrk", "syrk_finish", "allreduce", "spd_solve", "residual", "sumsq"):
                    ms, c = ctx.timer_get(k)
                    if c:
                        scopes[k] = round(ms / c, 5)
        ctx.timer_enable(False)
        X, lam, chi, acc, rej = out
        print("%s m=%d n=%d ms/iteration: timers off %.4f (%.1f iterations/s), on %.4f; scopes %s sum %.4f; acc %d rej %d chi %.6e lam %g "
              "xsum %.17g" % (name, m, n, res[False], 1e3 / res[False], res[True], scopes, sum(scopes.values()), acc, rej, chi, lam,
                              float(np.sum(X))))
    ctx.free(Jd); ctx.free(Fd); ctx.free(Ft); ctx.free(JTJd)
    del f
