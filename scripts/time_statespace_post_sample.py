"""Time of the joint posterior draws of the state-space fit state (StateSpaceFitState.sample, gpcc_ss_state_sample) on one
GPU, beside the dense route.

  1. sample at N = 6144, 98 304, 393 216, NT = 1 000 and 70 000 test times, nsamples = 1 and 64 (generator deviates), with
     the records already built (one call before the timed ones), and the first call on a fresh state (records included);
  2. the dense route at N = 6144: fit_state + predict(full_cov=True), then a host Cholesky draw of the NT x NT covariance.
Matern52, three equal bands of synthetic data, test times uniform over the span.  Every call is synchronous (it copies the
draws to the host), so a host clock around it measures the call (median of the repeats after one warm-up).  The card's name,
power limit and maximum SM clock are read in the same run (nvidia-smi --query-gpu, read-only).
Usage: time_statespace_post_sample.py [--out profiles/statespace_post_sample_timing_r1.log] [--quick]"""
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
    ap.add_argument("--out", default=os.path.join("profiles", "statespace_post_sample_timing_r1.log"))
    ap.add_argument("--quick", action="store_true", help="small sizes only (rehearsal)")
    a = ap.parse_args()
    lines = []

    def emit(s):
        print(s, flush=True)
        lines.append(s)

    emit("card: " + card())
    ctx = gpcc_b200.Context(1)
    alpha, rho = np.array([1.2, 0.9, 1.6]), 7.0
    rng = np.random.default_rng(2)
    emit("%-8s %-7s %-10s %-34s %8s %12s" % ("N", "NT", "method", "call", "nsamples", "median ms"))
    for N in ([6144] if a.quick else [6144, 98304, 393216]):
        span = N / 6144 * 150.0
        t, y, s, d = synthetic.synthetic_bands([N // 3] * 3, seed=4, span=span)
        p = gpcc_b200.Problem(t, y, s, gpcc_b200.matern52, ctx, method="statespace")
        for NT in (1000, 70000):
            tt = [rng.uniform(0.0, span, n) for n in (NT // 3, NT // 3, NT - 2 * (NT // 3))]

            def first():
                st = p.statespace_fit_state(d, alpha, rho)
                t0 = time.perf_counter()
                st.sample(tt, 1, nsamples=1)
                ms = (time.perf_counter() - t0) * 1e3
                st.close()
                return ms
            first()
            emit("%-8d %-7d %-10s %-34s %8d %12.3f" % (N, NT, "ss", "first sample on a new state", 1,
                                                       float(np.median([first() for _ in range(3)]))))
            st = p.statespace_fit_state(d, alpha, rho)
            for ns in (1, 64):
                reps = 10 if N <= 98304 else 3
                ms = timed(lambda: st.sample(tt, 1, nsamples=ns), reps)
                emit("%-8d %-7d %-10s %-34s %8d %12.3f" % (N, NT, "ss", "sample (records built)", ns, ms))
            st.close()
        p.close()
    N = 6144
    t, y, s, d = synthetic.synthetic_bands([N // 3] * 3, seed=4, span=150.0)
    p = gpcc_b200.Problem(t, y, s, gpcc_b200.matern52, ctx)
    for NT in (1000,) if a.quick else (1000, 10000):
        tt = [rng.uniform(0.0, 150.0, n) for n in (NT // 3, NT // 3, NT - 2 * (NT // 3))]
        for ns in (1, 64):
            def dense():
                st = p.fit_state(d, alpha, rho)
                mu, _, S, _ = st.predict(tt, full_cov=True)
                c = np.linalg.cholesky(S)
                mu[None, :] + np.random.default_rng(1).standard_normal((ns, NT)) @ c.T
                st.close()
            emit("%-8d %-7d %-10s %-34s %8d %12.3f" % (N, NT, "dense", "fit_state + predict(full) + chol", ns,
                                                       timed(dense, 3)))
    p.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
