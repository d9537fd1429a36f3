"""Per-evaluation time of the dense and the state-space method (Problem(..., method="statespace")) on one GPU.

  1. logL and logL + gradient, both methods, at N = 1536, 6144, 12288 (matern52, three equal bands of cfg4-style data),
     batches of M = 1 and 1250 candidates;
  2. the state-space method alone at N = 49 152, 98 304, 393 216 (M = 1 and 1250);
  3. rank 0's fixed-theta share of the cfg4 grid (1250 candidates at N = 6144, as scripts/time_cfg4_share.py) with both
     methods.
Kernel time is the library's CUDA-event time (ms_eval_kernels); wall time includes the host.  The card's name, power limit
and maximum SM clock are read in the same run (nvidia-smi --query-gpu, read-only).  Usage:
time_statespace.py [--out profiles/statespace_timing_r1.log] [--quick]"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gpcc_b200  # noqa: E402
from gpcc_b200 import synthetic  # noqa: E402


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown (nvidia-smi failed)"


def batch(rng, M, d):
    delays = np.tile(d, (M, 1))
    delays[:, 1:] += rng.uniform(-3.0, 3.0, (M, 2))
    alpha = rng.uniform(0.8, 2.5, (M, 3))
    rho = rng.uniform(1.0, 30.0, M)
    return delays, alpha, rho


def timed(ctx, p, args, want_grad, reps):
    p.loglik_batch(*args, want_grad=want_grad)                # warm-up of this shape
    ms_k, t0 = 0.0, time.perf_counter()
    for _ in range(reps):
        p.loglik_batch(*args, want_grad=want_grad)
        ms_k += ctx.stats()["ms_eval_kernels"]
    wall = (time.perf_counter() - t0) * 1e3 / reps
    return wall, ms_k / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "statespace_timing_r1.log"))
    ap.add_argument("--quick", action="store_true", help="small sizes only (rehearsal)")
    a = ap.parse_args()
    lines = []

    def emit(s):
        print(s, flush=True)
        lines.append(s)

    emit("card: " + card())
    ctx = gpcc_b200.Context(1, profiling=True)
    rng = np.random.default_rng(1)
    both = [1536] if a.quick else [1536, 6144, 12288]
    ss_only = [] if a.quick else [49152, 98304, 393216]
    emit("%-8s %-10s %-6s %-5s %12s %12s %14s" % ("N", "method", "M", "grad", "wall ms", "kernel ms", "kernel us/eval"))
    for N in both + ss_only:
        t, y, s, d = synthetic.synthetic_bands([N // 3] * 3, seed=4, span=N / 6144 * 150.0)
        methods = ["dense", "statespace"] if N in both else ["statespace"]
        for method in methods:
            p = gpcc_b200.Problem(t, y, s, gpcc_b200.matern52, ctx, method=method)
            for M in (1, 1250):
                args = batch(rng, M, d)
                for g in (False, True):
                    if method == "dense" and M == 1250 and N > 6144:
                        continue                          # minutes per point; the M = 1 time scales
                    reps = 3 if (method == "dense" and N >= 6144) or N > 100000 else 5
                    wall, k = timed(ctx, p, args, g, reps)
                    emit("%-8d %-10s %-6d %-5d %12.3f %12.3f %14.3f" % (N, method, M, g, wall, k, k * 1e3 / M))
            p.close()
    # cfg4 share
    t4, y4, s4, _ = synthetic.synthetic_bands([2048, 2048, 2048], seed=4)
    c4 = np.arange(0.0, 19.8001, 0.2)
    grid4 = np.array([[0.0, x, z] for z in c4 for x in c4])
    d4 = grid4[np.arange(0, len(grid4), 8)][:40 if a.quick else 1250]
    th4 = np.concatenate([np.log(np.expm1(np.array([1.0, 2.2, 4.0]))), [np.log((3.5 - 0.1) / (300.0 - 3.5))]])[None]
    res = {}
    for method in ("dense", "statespace"):
        p4 = gpcc_b200.Problem(t4, y4, s4, gpcc_b200.matern52, ctx, method=method)
        p4.grid_posterior(d4[:40], th4, iterations=0, rhomin=0.1, rhomax=300.0)
        t0 = time.perf_counter()
        r = p4.grid_posterior(d4, th4, iterations=0, rhomin=0.1, rhomax=300.0)
        dt = time.perf_counter() - t0
        res[method] = r["loglikel"]
        emit("cfg4 share, %-10s: %d candidates, %.3f s wall, kernel %.3f s, %.3f ms per candidate, path %d" % (
            method, len(d4), dt, ctx.stats()["ms_eval_kernels"] * 1e-3, dt * 1e3 / len(d4), ctx.stats()["path"]))
        p4.close()
    emit("cfg4 share: max |logL(statespace) - logL(dense)| / |logL| = %.3e" % np.max(
        np.abs(res["statespace"] - res["dense"]) / np.abs(res["dense"])))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
