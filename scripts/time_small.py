"""Kernel-time probe of the fused small-N kernel (dev script)."""
import sys, os
import numpy as np
sys.path.insert(0, ".")
import oracle
from gpcc_b200 import Problem, Context
ctx = Context(1, profiling=True)
M = 148 * int(os.environ.get("GPCC_TS_WAVES", "64"))
rg = np.random.default_rng(1)
delays = np.zeros((M, 3)); delays[:, 1:] = rg.uniform(0, 20, (M, 2))
alpha = rg.uniform(0.5, 3.0, (M, 3)); rho = rg.uniform(0.5, 20, M)
t, y, s, d = oracle.simulatethreelightcurves()
for nb, N in ((3, 150), (2, 110)):
    p = Problem(t[:nb], y[:nb], s[:nb], "matern32", ctx)
    op = oracle.Problem(t[:nb], y[:nb], s[:nb], "matern32")
    for it in range(3):
        ll, g, info = p.loglik_batch(delays[:, :nb], alpha[:, :nb], rho, want_grad=True)
        st = ctx.stats()
    for it in range(3):
        ll0, info0 = p.loglik_batch(delays[:, :nb], alpha[:, :nb], rho)
        st0 = ctx.stats()
    assert np.array_equal(ll0, ll), np.max(np.abs(ll0 - ll))
    print("   logL only (forward-only): kernel %.3f ms  %.1f us/eval-slot  %.2f TFLOP/s (N^3/3)" % (
        st0["ms_eval_kernels"], st0["ms_eval_kernels"] * 1e3 / (M / 148),
        M * float(N)**3 / 3 / st0["ms_eval_kernels"] / 1e9), flush=True)
    r = [op.loglik_grad(delays[m, :nb], alpha[m, :nb], rho[m]) for m in range(8)]
    err = max(abs(ll[m] - r[m][0]) / abs(r[m][0]) for m in range(8)); gerr = max(np.max(np.abs(g[m] - r[m][1])) for m in range(8))
    print("variant", os.environ.get("GPCC_SMALL_VARIANT", "0"), "N=%d" % N, "kernel %.3f ms  %.1f us/eval-slot  %.2f TFLOP/s (N^3)  relerr %.1e graderr %.1e" % (
        st["ms_eval_kernels"], st["ms_eval_kernels"] * 1e3 / (M / 148), M * float(N)**3 / st["ms_eval_kernels"] / 1e9, err, gerr), flush=True)
