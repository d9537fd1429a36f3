#!/usr/bin/env python
"""bench.py -- delay candidates/sec (fitted logL+grad) of the B200-native GPCC hot path.

A "step" is one pass of the hot path over one batch of synthetic input: fit every candidate of a delay grid (5 screening
evaluations + L-BFGS on the analytic gradient, all of it inside one persistent CUDA kernel per GPU), all-gather the
per-candidate results across the GPUs (the library's own ncclAllGather) and normalise the log-likelihoods into the
posterior under the delay prior -- `gpcc_grid_posterior`, the call that replaces the README's `pmap` + `getprobabilities`.
Workload = BASELINE.json configs[2] (simulatethreelightcurves-style data, 2-D grid (0:0.2:20)^2 = 10 201 candidates,
matern32, rhomax=300, iterations=1000) -- the configuration the metric "candidates/sec at 1/2/4/8 B200" is quoted on.
Default scaling is STRONG: the one 10 201-candidate grid is sharded over the N ranks (north_star: "sharding the grid
across the 8 GPUs").  `--scaling weak` refines the grid N-fold (10 201 candidates per GPU); at N > 1 the other mode is
reported under "also".  configs[1] (101 candidates) cannot occupy 148 SMs and configs[3] (N=6144) is a fixed-theta
sweep; both are reported under "also".

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--scaling strong|weak] [--workload cfg3|cfg2]
                  [--dump-outputs DIR]

--dump-outputs DIR writes what the last timed step returned (every array of the `grid_posterior` result) as DIR/<name>.npy
in float64.  The workload is seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

RHOMIN, RHOMAX, ITERATIONS, INITIALRANDOM = 0.1, 300.0, 1000, 5
METRIC = "delay candidates/sec (fitted logL+grad)"


def make_workload(name, refine=1):
    """Returns (tarray, yarray, sarray, delays[M][L], label).  Data generator: gpcc_b200.synthetic (host, numpy).
    refine > 1 (weak scaling): the grid is refined `refine`-fold along the last delay."""
    from gpcc_b200 import synthetic
    if name == "cfg3":
        t, y, s, _ = synthetic.simulatethreelightcurves()
        c2 = np.arange(0.0, 20.0001, 0.2)
        c3 = np.linspace(0.0, 20.0, 101 * refine)
        delays = np.array([[0.0, a, b] for b in c3 for a in c2])          # d1 fastest (README.md:231-235)
        label = "cfg3: simulatethreelightcurves-style N=(60,50,40), grid (0:0.2:20) x %d points in [0,20] = %d candidates, matern32" % (len(c3), len(delays))
    elif name == "cfg2":
        t, y, s, _ = synthetic.simulatetwolightcurves()
        c = np.linspace(0.0, 10.0, 101 * refine) if refine > 1 else np.arange(0.0, 10.0001, 0.1)
        delays = np.stack([np.zeros_like(c), c], 1)
        label = "cfg2: simulatetwolightcurves-style N=(60,50), 1-D grid over [0,10] = %d candidates, matern32" % len(delays)
    else:
        raise SystemExit("unknown workload " + name)
    return t, y, s, delays, label


def common_config(label):
    """The keys both arms (ours / reference) report, so that the driver can tell they ran the same configuration."""
    return {"workload": label, "kernel": "matern32", "rhomin": RHOMIN, "rhomax": RHOMAX, "iterations": ITERATIONS,
            "initialrandom": INITIALRANDOM}


# ---- CPU baseline: the oracle (restated reference, Nelder-Mead like the reference) over a process pool -------------
_W = {}


def _cpu_init(tys, theta0):
    try:
        from threadpoolctl import threadpool_limits
        _W["lim"] = threadpool_limits(1)            # OpenBLAS pinned to 1 thread per worker (BASELINE.md section 4)
    except Exception:
        pass
    import oracle  # noqa: F401  (import cost paid before the first timed task)
    _W["tys"], _W["theta0"] = tys, theta0


def _cpu_fit(dl):
    import oracle
    t, y, s = _W["tys"]
    return oracle.gpcc(t, y, s, kernel="matern32", delays=dl, iterations=ITERATIONS, rhomin=RHOMIN, rhomax=RHOMAX,
                       theta0=_W["theta0"][None], optimizer="neldermead")[0]


def cpu_reference_rate(t, y, s, delays, theta0, steps=1, warmup=1, per_core=4):
    """README `pmap` recipe (README.md:185-206) on the host cores with the oracle: one candidate per task, workers = all
    cores, OpenBLAS pinned to one thread per worker.  Sample = per_core x cores candidates evenly spaced over the grid; every
    warm-up step is a full pass over the sample (so that every worker has imported, paged in and run the code before the
    clock starts).  Returns (candidates/s, cores, sample size, [seconds per step])."""
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    idx = np.unique(np.linspace(0, len(delays) - 1, per_core * cores).astype(int))
    sample = delays[idx]
    ctxmp = mp.get_context("fork")
    times = []
    with ctxmp.Pool(cores, initializer=_cpu_init, initargs=((t, y, s), theta0)) as pool:
        for _ in range(max(warmup, 1)):
            pool.map(_cpu_fit, sample, chunksize=1)
        for _ in range(steps):
            t0 = time.perf_counter()
            pool.map(_cpu_fit, sample, chunksize=1)
            times.append(time.perf_counter() - t0)
    return len(sample) / float(np.mean(times)), cores, len(sample), times


def cpu_sample_text(ns, M, cores):
    return ("%d of %d candidates (evenly spaced over the grid) per step, one candidate per task, pool of %d processes x 1 BLAS "
            "thread, oracle = restated reference with Nelder-Mead g_tol=1e-6 (the reference's optimiser)" % (ns, M, cores))


def dump_outputs(outdir, res):
    """One .npy per array of a grid_posterior result; the integer counters (nfev, info) are widened to float64.  The cfg3
    grid gives 11 doubles per candidate: 0.9 MB, 7 MB at 8-fold weak scaling."""
    os.makedirs(outdir, exist_ok=True)
    for name, a in res.items():
        np.save(os.path.join(outdir, name + ".npy"), np.asarray(a, dtype=np.float64))


class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(np.max(mx)) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def run_reference(args, rank, out):
    """--impl reference: the reference's own CPU path (restated: no Julia in this image) on the host cores."""
    if rank != 0:
        return
    t, y, s, delays, label = make_workload(args.workload, 1)
    import gpcc_b200
    theta0 = gpcc_b200.initial_solutions(y, 1, 1, INITIALRANDOM, RHOMIN, RHOMAX)[0][0]
    rate, cores, ns, times = cpu_reference_rate(t, y, s, delays, theta0, steps=args.steps, warmup=args.warmup, per_core=args.cpu_per_core)
    line = {"impl": "reference", "metric": METRIC, "value": rate, "unit": "candidates/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": float(np.mean(times)) * 1e3, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": common_config(label),
            "details": {"optimizer": "Nelder-Mead g_tol=1e-6 (the reference's), iterations=1000, initialrandom=5",
                        "note": "restated reference (numpy/scipy oracle), not Julia: no julia toolchain in this image",
                        "step_seconds_min_max": [float(np.min(times)), float(np.max(times))]},
            "cpu_baseline": {"value": rate, "unit": "candidates/s", "cores": cores, "kind": "port", "sample": cpu_sample_text(ns, len(delays), cores)},
            "e2e": {"value": rate, "unit": "candidates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    out.write(json.dumps(line) + "\n")
    out.flush()


def run_single_process(args, out):
    """One process, N devices: gpcc_ctx_create(ndev=N) -> one host thread per device, ncclCommInitAll + ncclAllGather inside the
    library (what the Julia shim's default context does with GPCC_B200_NDEV=N).  Same workload and step as the default mode."""
    import torch
    import gpcc_b200
    t, y, s, delays, label = make_workload(args.workload, args.gpus if args.scaling == "weak" else 1)
    theta0 = gpcc_b200.initial_solutions(y, 1, 1, INITIALRANDOM, RHOMIN, RHOMAX)[0][0]
    ctx = gpcc_b200.Context(ndev=args.gpus, profiling=True)
    problem = gpcc_b200.Problem(t, y, s, gpcc_b200.matern32, ctx)
    flush = [torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda:%d" % d) for d in range(args.gpus)]
    def sync():
        for d in range(args.gpus):
            torch.cuda.synchronize(d)
    for _ in range(max(args.warmup, 3)):
        problem.grid_posterior(delays, theta0, iterations=ITERATIONS, rhomin=RHOMIN, rhomax=RHOMAX)
    times = []
    for i in range(args.steps):
        for f in flush:
            f.fill_(float(i))
        sync()
        t0 = time.perf_counter()
        res = problem.grid_posterior(delays, theta0, iterations=ITERATIONS, rhomin=RHOMIN, rhomax=RHOMAX)   # synchronous call
        times.append(time.perf_counter() - t0)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, res)
    st = ctx.stats()
    ms = float(np.mean(times)) * 1e3
    line = {"metric": METRIC, "value": len(delays) / (ms * 1e-3), "unit": "candidates/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": common_config(label),
            "details": {"mode": "single process, gpcc_ctx_create(ndev=%d): one host thread per device, ncclCommInitAll + ncclAllGather in the library" % args.gpus,
                        "timing": "host wall clock around the synchronous call (devices idle before and after), L2 flushed between steps",
                        "kernel_ms_per_step_max_over_devices": st["ms_eval_kernels"], "posterior_sum": float(np.sum(res["posterior"]))}}
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    # stdout must carry exactly ONE JSON line: libraries (NCCL prints its version banner) write to fd 1, so fd 1 is
    # pointed at stderr for the duration of the run and the JSON line is written to the saved descriptor.
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=["cfg3", "cfg2"])
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--cpu-per-core", type=int, default=4, help="candidates per host core in the CPU sample")
    ap.add_argument("--single-process", action="store_true",
                    help="one process driving --gpus N devices through gpcc_ctx_create(ndev=N) (the layout a single Julia process uses) instead of one rank per GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-also", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the library's timed step; --impl reference has none")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, real_stdout)
        return
    if args.single_process:
        return run_single_process(args, real_stdout)
    if world != args.gpus and world > 1:
        raise SystemExit("--gpus must equal WORLD_SIZE under torchrun")
    if args.gpus > 1 and world == 1:
        raise SystemExit("for --gpus N>1 launch with python -m torch.distributed.run --nproc-per-node N bench.py --gpus N ...")
    warmup = max(args.warmup, 3)

    import gpcc_b200
    t, y, s, delays, label = make_workload(args.workload, world if args.scaling == "weak" else 1)
    theta0 = gpcc_b200.initial_solutions(y, 1, 1, INITIALRANDOM, RHOMIN, RHOMAX)[0][0]
    M = len(delays)

    # ---- CPU baseline first (fork before any CUDA state exists), rank 0 at N=1 only; same sampling as --impl reference ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        rate, cores, ns, times = cpu_reference_rate(t, y, s, delays, theta0, steps=1, warmup=1, per_core=args.cpu_per_core)
        cpu = {"value": rate, "unit": "candidates/s", "cores": cores, "kind": "port", "sample": cpu_sample_text(ns, M, cores) + ", %.1f s" % times[0]}

    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    ctx = gpcc_b200.Context(devices=[local_rank], profiling=True)
    if world > 1:
        # the library owns the collective on the path: rank 0 draws the NCCL id, torch.distributed only carries its 128 bytes
        box = [gpcc_b200.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        ctx.comm_init_rank(world, rank, box[0])
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)     # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        e0 = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
        e1 = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
        wall = 0.0
        for i in range(steps):
            flush.fill_(float(i))              # L2 flush between timed iterations (untimed)
            barrier()
            e0[i].record()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            e1[i].record()
            wall += time.perf_counter() - t0
            barrier()
        if os.environ.get("GPCC_BENCH_VERBOSE"):
            sys.stderr.write("rank %d %s per-step ms: %s\n" % (rank, fn.__name__, ["%.0f" % a.elapsed_time(b) for a, b in zip(e0, e1)]))
        dev_ms = sum(a.elapsed_time(b) for a, b in zip(e0, e1))
        tmax = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        return float(tmax.item()) / steps, wall * 1e3 / steps

    def measure(delays_, label_):
        """Times the resident and the end-to-end step on the grid `delays_`; returns the pieces of the JSON line."""
        problem = gpcc_b200.Problem(t, y, s, gpcc_b200.matern32, ctx)
        state, kstats = {}, []

        def step_resident():
            res = problem.grid_posterior(delays_, theta0, iterations=ITERATIONS, rhomin=RHOMIN, rhomax=RHOMAX)
            kstats.append(ctx.stats())
            state.update(res=res)
            return res["posterior"]

        def step_e2e():
            # the user-facing call with HOST buffers: upload the light curves, fit the grid, posterior back on the host
            pr = gpcc_b200.Problem(t, y, s, gpcc_b200.matern32, ctx)
            res = pr.grid_posterior(delays_, theta0, iterations=ITERATIONS, rhomin=RHOMIN, rhomax=RHOMAX)
            state.update(stats_e2e=ctx.stats())
            pr.close()
            return res["posterior"]

        for _ in range(warmup):
            step_resident()
        del kstats[:]
        ms_step, wall_ms = timed(step_resident, args.steps)
        for _ in range(2):
            step_e2e()
        ms_e2e, _ = timed(step_e2e, args.steps)
        problem.close()
        return dict(ms_step=ms_step, wall_ms=wall_ms, ms_e2e=ms_e2e, kstats=list(kstats), state=state, M=len(delays_), label=label_)

    sampler = ClockSampler(local_rank)
    if rank == 0 and not os.environ.get("GPCC_BENCH_NO_SAMPLER"):
        sampler.start()
    r = measure(delays, label)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, r["state"]["res"])      # every rank holds the full, all-gathered result

    # ---- roofline of the dominant kernel (persistent fit kernel = fused small-N evaluator), from the library's CUDA events ----
    N = int(sum(len(a) for a in t))
    L = len(t)
    ks = r["kstats"]
    n_grad = sum(k["n_evals_grad"] for k in ks)
    n_fwd = sum(k["n_evals"] - k["n_evals_grad"] for k in ks)
    kern_ms = sum(k["ms_eval_kernels"] for k in ks)
    n_launch = sum(k["n_eval_launches"] for k in ks)
    peaks = json.load(open(os.path.join(ROOT, "profiles", "fp64_peaks_r1.json")))
    flops = n_grad * float(N) ** 3 + n_fwd * float(N) ** 3 / 3.0          # algorithmic: N^3 per logL+grad, N^3/3 per logL-only evaluation
    achieved = flops / (kern_ms * 1e-3) / 1e12
    traffic = None
    tp = os.path.join(ROOT, "profiles", "small_fit_traffic.json")
    if os.path.exists(tp):
        traffic = json.load(open(tp)).get("dram_bytes_per_launch")
    roofline = {"bound": "tensor", "pipe": "FP64 DFMA pipe (the kernel issues scalar DFMA; on B200 the DMMA tensor peak is the same: 37.0 vs 36.7 TFLOP/s measured)",
                "kernel": "small_fit_kernel (persistent: screening + L-BFGS + fused assembly / symmetric sweep / gradient, one CTA per candidate)",
                "achieved": achieved, "peak": peaks["dfma_tflops"], "unit": "TFLOP/s", "frac": achieved / peaks["dfma_tflops"],
                "traffic": traffic, "peak_source": "measured, profiles/fp64_peaks_r1.json (MEASURED_PEAKS.json has no FP64 entry)",
                "algorithmic_flops": "N^3 per logL+gradient evaluation, N^3/3 per forward-only (screening) evaluation, N=%d" % N,
                "grad_evals_per_step": n_grad / args.steps, "forward_evals_per_step": n_fwd / args.steps,
                "kernel_ms_per_step": kern_ms / args.steps, "kernel_share_of_step": kern_ms / args.steps / r["ms_step"]}

    nfev = r["state"]["res"]["nfev"]
    rec = (L + 1 + 4) * 8                                   # per-candidate record of the all-gather / result download
    data_bytes = N * (4 * 8 + 4)
    M_local = (M + world - 1) // world
    line = {"metric": METRIC, "value": M / (r["ms_step"] * 1e-3), "unit": "candidates/s", "n_gpus": world, "steps": args.steps,
            "warmup": warmup, "ms_per_step": r["ms_step"], "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": common_config(label),
            "details": {"optimizer": "L-BFGS (m=8) on the analytic gradient, device resident: one persistent CTA per candidate (small_fit.cu)",
                        "candidates_per_gpu": M_local, "l2": "256 MB flush buffer written between timed steps",
                        "parallelism": "candidate m on rank m mod %d; one ncclAllGather (library-owned communicator) of the per-candidate records, log-sum-exp on device" % world,
                        "mean_nfev": float(np.mean(nfev)), "max_nfev": int(np.max(nfev))},
            "e2e": {"value": M / (r["ms_e2e"] * 1e-3), "unit": "candidates/s",
                    "h2d_bytes_per_step": int(data_bytes + M_local * L * 8 + INITIALRANDOM * (L + 1) * 8 + (M_local * rec if world > 1 else M * 8)),
                    "d2h_bytes_per_step": int(M_local * ((L + 1) * 8 + 8 + 12) + (world * M_local * (rec + 8) if world > 1 else M * 8)),
                    "ms_per_step": r["ms_e2e"]},
            "gpu_launches": int(n_launch), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
            "wall_ms_per_step": r["wall_ms"]}

    also = {}
    if not args.no_also and args.workload == "cfg3":
        if world > 1:
            # the other scaling mode, for the record
            other = "weak" if args.scaling == "strong" else "strong"
            t_, y_, s_, d_o, l_o = make_workload("cfg3", world if other == "weak" else 1)
            ro = measure(d_o, l_o)
            also["scaling_" + other] = {"workload": l_o, "candidates_per_s": len(d_o) / (ro["ms_step"] * 1e-3), "ms_per_step": ro["ms_step"],
                                        "e2e_candidates_per_s": len(d_o) / (ro["ms_e2e"] * 1e-3)}
        # configs[3] (3 bands x 2048 points, N=6144, matern52): the tiled large-N path on the north-star workload, a fixed-theta
        # posterior over the 100 x 100 delay grid (0:0.2:19.8)^2, one blocked Cholesky (N^3/3 flop, DMMA trailing updates) per
        # candidate (iterations=0: screening only).  Every rank takes 1 250 candidates (its share of the 8-GPU run), so at 8 GPUs
        # this IS the full 10^4-candidate grid of the "< 10 s" target and below it is the share of the first N ranks of that run.
        try:
            from gpcc_b200 import synthetic
            t4, y4, s4, _ = synthetic.synthetic_bands([2048, 2048, 2048], seed=4)
            p4 = gpcc_b200.Problem(t4, y4, s4, gpcc_b200.matern52, ctx)
            c4 = np.arange(0.0, 19.8001, 0.2)
            grid4 = np.array([[0.0, a, b] for b in c4 for a in c4])
            share = int(os.environ.get("GPCC_BENCH_CFG4_SHARE", "1250"))
            # below 8 GPUs: the candidates that ranks 0 .. world-1 own in the 8-GPU run (candidate m -> rank m mod 8), in grid order, so
            # that rank j of this run works on exactly the share of rank j of the full run (runs of 50 candidates with a common
            # tau_2), not on a corner of the grid with 12-candidate stubs
            sel4 = np.array([m for m in range(len(grid4)) if m % 8 < min(world, 8)])
            d4 = grid4[sel4][: share * world]
            th4 = np.concatenate([np.log(np.expm1(np.array([1.0, 2.2, 4.0]))), [np.log((3.5 - RHOMIN) / (RHOMAX - 3.5))]])[None]
            p4.grid_posterior(d4[: 40 * world], th4, iterations=0, rhomin=RHOMIN, rhomax=RHOMAX)            # warm-up: a full wave of 32 matrices per rank, so that the workspace and the last-band cache have their final size (a 16-candidate warm-up left a 5 GB re-allocation, 0.1-0.7 s, inside the timed call)
            barrier()
            t0 = time.perf_counter()
            r4 = p4.grid_posterior(d4, th4, iterations=0, rhomin=RHOMIN, rhomax=RHOMAX)
            torch.cuda.synchronize()
            dt4 = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(dt4, op=dist.ReduceOp.MAX)
            dt4 = float(dt4.item())
            st4 = ctx.stats()
            fl = share * float(6144) ** 3 / 3.0
            # executed flops on the N^3/3 model (n = 2048 points per band): an evaluation that took the leading 2n x 2n block from its wave
            # saves (2n)^3/3; one that imported the band-1 steps of its last band from the last-band cache saves 2 n^3 (the solve
            # L31 = K31 L11^-T and the update K33 - L31 L31'), which every distinct tau_3 on this rank pays once
            n_tau3 = len(np.unique(d4[rank::world][:, 2])) if st4["n_tau_cache"] else 0
            fl_exec = fl - st4["n_shared_prefix"] * float(4096) ** 3 / 3.0 - (st4["n_tau_cache"] - n_tau3) * 2.0 * float(2048) ** 3
            hbm = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"] if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else 6650.0
            also["cfg4"] = {"workload": "3 bands x 2048 points (N=6144), matern52, fixed-theta posterior over %d candidates of the 100x100 grid (0:0.2:19.8)^2, %d per GPU" % (len(d4), share),
                            "seconds": dt4, "candidates_per_s": len(d4) / dt4, "ms_per_candidate_per_gpu": dt4 * 1e3 / share,
                            "structure_reuse": "%d of %d evaluations on this rank took their leading 4096 x 4096 block (bands 1-2: same tau_2) from another evaluation of their wave; %d took the band-1 steps of band 3 (a function of tau_3 alone) from the last-band cache, filled once for each of the %d distinct tau_3" % (st4["n_shared_prefix"], share, st4["n_tau_cache"], n_tau3),
                            "cholesky_effective_tflops_per_gpu": fl / (st4["ms_factor"] * 1e-3) / 1e12,
                            "cholesky_executed_tflops_per_gpu": fl_exec / (st4["ms_factor"] * 1e-3) / 1e12,
                            "cholesky_frac_of_fp64_peak": fl_exec / (st4["ms_factor"] * 1e-3) / 1e12 / peaks["dmma_m8n8k4_tflops"],
                            "cholesky_flop_model": "effective = algorithmic N^3/3 per candidate; executed = that minus (4096)^3/3 for every evaluation that took the leading block from its wave and minus 2 x 2048^3 for every evaluation served by the last-band cache (plus its fills); the fraction of peak is quoted on the EXECUTED flops",
                            "assembly_GBps": st4["assembly_bytes"] / (st4["ms_assembly"] * 1e-3) / 1e9,
                            "assembly_frac_of_hbm_peak": st4["assembly_bytes"] / (st4["ms_assembly"] * 1e-3) / 1e9 / hbm,
                            "assembly_bytes_model": "bytes the assembly kernels moved on this rank as counted by the library (tiles written, 131 072 B each; block (3,3) imported from the last-band cache counts read + written; shared and cached tiles are not assembled at all), %.1f MB per candidate against 4 N (N+1) = %.1f MB for a full lower triangle" % (st4["assembly_bytes"] / share / 1e6, 4.0 * 6144 * 6145 / 1e6),
                            "posterior_sum": float(np.sum(r4["posterior"])),
                            "north_star_target": "8 GPUs x 1250 = the full 10^4-candidate grid in < 10 s" + (": measured %.2f s" % dt4 if world == 8 else " (projected from this run: %.2f s)" % dt4)}
            p4.close()
        except Exception as e:      # never lose the headline line over the side measurement
            also["cfg4"] = {"error": repr(e)}
        if rank == 0 and world == 1:
            # The same grid with the REFERENCE'S OWN optimiser on the device (Nelder-Mead, g_tol 1e-6, forward-only evaluations):
            # the like-for-like counterpart of the CPU baseline / --impl reference arm, which also runs Nelder-Mead.  The headline
            # uses L-BFGS on the analytic gradient as north_star specifies (~12x fewer evaluations).
            pn = gpcc_b200.Problem(t, y, s, gpcc_b200.matern32, ctx)
            pn.grid_posterior(delays, theta0, iterations=ITERATIONS, rhomin=RHOMIN, rhomax=RHOMAX, optimizer="neldermead")
            t0 = time.perf_counter()
            rn = pn.grid_posterior(delays, theta0, iterations=ITERATIONS, rhomin=RHOMIN, rhomax=RHOMAX, optimizer="neldermead")
            dtn = time.perf_counter() - t0
            also["cfg3_neldermead"] = {"workload": label, "optimizer": "Nelder-Mead (Optim.jl's adaptive variant, g_tol=1e-6) as a device state machine",
                                       "candidates_per_s": M / dtn, "seconds_per_grid": dtn, "mean_evaluations": float(np.mean(rn["nfev"])),
                                       "max_abs_posterior_difference_to_lbfgs": float(np.max(np.abs(rn["posterior"] - r["state"]["res"]["posterior"])))}
            pn.close()
            # configs[1] (101 candidates, 2 bands) for the record
            t2, y2, s2, d2, label2 = make_workload("cfg2", 1)
            p2 = gpcc_b200.Problem(t2, y2, s2, gpcc_b200.matern32, ctx)
            th2 = gpcc_b200.initial_solutions(y2, 1, 1, INITIALRANDOM, RHOMIN, RHOMAX)[0][0]
            for _ in range(3):
                p2.grid_posterior(d2, th2, iterations=ITERATIONS, rhomin=RHOMIN, rhomax=RHOMAX)
            t0 = time.perf_counter()
            for _ in range(5):
                p2.grid_posterior(d2, th2, iterations=ITERATIONS, rhomin=RHOMIN, rhomax=RHOMAX)
            dt = (time.perf_counter() - t0) / 5
            also["cfg2"] = {"workload": label2, "candidates_per_s": len(d2) / dt, "ms_per_grid": dt * 1e3}
    if also:
        line["also"] = also
    if rank == 0:
        real_stdout.write(json.dumps(line) + "\n")
        real_stdout.flush()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
