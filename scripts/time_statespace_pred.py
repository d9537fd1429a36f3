"""Time of the state-space fit state (Problem.statespace_fit_state, gpcc_ss_state_*) on one GPU, beside the dense fit state.

  1. state creation (forward filter that stores its moments + backward pass) at N = 6144, 98 304, 393 216;
  2. predict (means and standard deviations) at NT = 1000 and 70 000 test points, predict_loglik at NT = 1000;
  3. the dense fit_state (one Cholesky factorisation of K + Sobs) + predict at NT = 1000, N = 6144 and 12 288.
Matern52, three equal bands of synthetic data.  Every call is synchronous, so a host clock around it measures the call
(median of the repeats after one warm-up).  The card's name, power limit and maximum SM clock are read in the same run
(nvidia-smi --query-gpu, read-only).  Usage: time_statespace_pred.py [--out profiles/statespace_pred_timing_r1.log] [--quick]"""
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
    ap.add_argument("--out", default=os.path.join("profiles", "statespace_pred_timing_r1.log"))
    ap.add_argument("--quick", action="store_true", help="small sizes only (rehearsal)")
    a = ap.parse_args()
    lines = []

    def emit(s):
        print(s, flush=True)
        lines.append(s)

    emit("card: " + card())
    ctx = gpcc_b200.Context(1)
    rng = np.random.default_rng(1)
    alpha, rho = np.array([1.2, 0.9, 1.6]), 7.0
    emit("%-8s %-10s %-16s %8s %12s" % ("N", "state", "call", "NT", "median ms"))
    for N in ([6144] if a.quick else [6144, 98304, 393216]):
        t, y, s, d = synthetic.synthetic_bands([N // 3] * 3, seed=4, span=N / 6144 * 150.0)
        p = gpcc_b200.Problem(t, y, s, gpcc_b200.matern52, ctx, method="statespace")
        reps = 3 if N > 100000 else 5
        emit("%-8d %-10s %-16s %8s %12.3f" % (N, "ss", "create", "-", timed(lambda: p.statespace_fit_state(d, alpha, rho).close(), reps)))
        st = p.statespace_fit_state(d, alpha, rho)
        lo, hi = min(x.min() for x in t), max(x.max() for x in t)
        for NT in (1000, 70000):
            tt = [rng.uniform(lo, hi, NT // 3 + (1 if l < NT % 3 else 0)) for l in range(3)]
            emit("%-8d %-10s %-16s %8d %12.3f" % (N, "ss", "predict", NT, timed(lambda: st.predict(tt), 10)))
        tt = [rng.uniform(lo, hi, n) for n in (334, 333, 333)]
        yt = [np.full(len(x), np.mean(yy)) for x, yy in zip(tt, y)]
        sg = [0.5 * np.ones(len(x)) for x in tt]
        emit("%-8d %-10s %-16s %8d %12.3f" % (N, "ss", "predict_loglik", 1000, timed(lambda: st.predict_loglik(tt, yt, sg), reps)))
        st.close()
        p.close()
    for N in ([6144] if a.quick else [6144, 12288]):
        t, y, s, d = synthetic.synthetic_bands([N // 3] * 3, seed=4, span=N / 6144 * 150.0)
        p = gpcc_b200.Problem(t, y, s, gpcc_b200.matern52, ctx)
        lo, hi = min(x.min() for x in t), max(x.max() for x in t)
        tt = [rng.uniform(lo, hi, n) for n in (334, 333, 333)]
        emit("%-8d %-10s %-16s %8s %12.3f" % (N, "dense", "create", "-", timed(lambda: p.fit_state(d, alpha, rho).close(), 3)))
        st = p.fit_state(d, alpha, rho)
        emit("%-8d %-10s %-16s %8d %12.3f" % (N, "dense", "predict", 1000, timed(lambda: st.predict(tt), 3)))
        st.close()
        p.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
