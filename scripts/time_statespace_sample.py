"""Time of the O(N) state-space draw (Problem.statespace_sample, gpcc_ss_sample) on one GPU, beside the dense draw.

  1. statespace_sample at N = 6144, 98 304, 393 216 and 1 048 576, nsamples = 1 and 64 (deviates from the generator);
  2. the dense fit_state (one Cholesky factorisation of K + Sobs) + sample at N = 6144, nsamples = 1 and 64.
Matern52, three equal bands of synthetic data.  Every call is synchronous (it copies the draws to the host), so a host clock
around it measures the call (median of the repeats after one warm-up).  The card's name, power limit and maximum SM clock
are read in the same run (nvidia-smi --query-gpu, read-only).
Usage: time_statespace_sample.py [--out profiles/statespace_sample_timing_r1.log] [--quick]"""
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


def timed(f, reps):
    f()                                                   # warm-up of this shape
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        f()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "statespace_sample_timing_r1.log"))
    ap.add_argument("--quick", action="store_true", help="small sizes only (rehearsal)")
    a = ap.parse_args()
    lines = []

    def emit(s):
        print(s, flush=True)
        lines.append(s)

    emit("card: " + card())
    ctx = gpcc_b200.Context(1)
    alpha, rho = np.array([1.2, 0.9, 1.6]), 7.0
    emit("%-8s %-10s %-22s %8s %12s" % ("N", "method", "call", "nsamples", "median ms"))
    for N in ([6144] if a.quick else [6144, 98304, 393216, 1048576]):
        t, y, s, d = synthetic.synthetic_bands([N // 3] * 3, seed=4, span=N / 6144 * 150.0)
        p = gpcc_b200.Problem(t, y, s, gpcc_b200.matern52, ctx, method="statespace")
        for ns in (1, 64):
            reps = 10 if N * ns <= 393216 else 3
            ms = timed(lambda: p.statespace_sample(d, alpha, rho, 1, nsamples=ns), reps)
            emit("%-8d %-10s %-22s %8d %12.3f" % (N, "ss", "statespace_sample", ns, ms))
        p.close()
    N = 6144
    t, y, s, d = synthetic.synthetic_bands([N // 3] * 3, seed=4, span=150.0)
    p = gpcc_b200.Problem(t, y, s, gpcc_b200.matern52, ctx)
    for ns in (1, 64):
        def dense():
            st = p.fit_state(d, alpha, rho)
            st.sample(1, ns)
            st.close()
        emit("%-8d %-10s %-22s %8d %12.3f" % (N, "dense", "fit_state + sample", ns, timed(dense, 3)))
    st = p.fit_state(d, alpha, rho)
    for ns in (1, 64):
        emit("%-8d %-10s %-22s %8d %12.3f" % (N, "dense", "sample (state built)", ns, timed(lambda: st.sample(1, ns), 5)))
    st.close()
    p.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
