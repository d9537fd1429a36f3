"""Every kernel variant the host dispatch can select, against the oracle and against each other (run with -m gpu on a B200).

The host code picks between separately compiled code paths: the fused small-N evaluator and the persistent fit kernel by
tile count T = ceil((N+1)/8) and by batch size relative to the SM count (with_instantiation in small_eval.cuh: <128,2>,
<128,3>, <192,2>, <224,1>, <352,1>); the tiled path by wave size (512, 128 or 32 matrices by N), look-ahead on two streams,
the shared leading block and the last-band cache (large_path.cu); the fitted state by tile edges of its triangular solve, Gram product
and one-CTA Cholesky (predict.cu).  A bug in one of them shows only in the calls that select it, so each is selected here
on purpose.  Tolerances are those of test_gpu_parity.py; "bitwise" means np.array_equal.
"""
import itertools
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest
import scipy.linalg as sla

import gpcc_b200
import oracle
from conftest import load_golden
from gpcc_b200 import Problem

pytestmark = pytest.mark.gpu

LL_RTOL = 1e-10
GRAD_RTOL = 1e-8
FIT_ATOL = 1e-6
PRED_RTOL = 1e-8
TESTS = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(TESTS)


@pytest.fixture(scope="module")
def nsm():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _split(N, nb, rg):
    """N points in nb bands of at least 2 points each, sizes drawn from rg."""
    extra = N - 2 * nb
    cuts = np.sort(rg.integers(0, extra + 1, nb - 1))
    return [int(v) + 2 for v in np.diff(np.r_[0, cuts, extra])]


def _bands(N, L=3):
    return [N // L + (1 if l < N % L else 0) for l in range(L)]


def _pack(t, y, s):
    return dict(t=np.concatenate(t), y=np.concatenate(y), s=np.concatenate(s), n=np.array([len(a) for a in t]))


def _unpack(z):
    idx = np.cumsum(z["n"])[:-1]
    return np.split(z["t"], idx), np.split(z["y"], idx), np.split(z["s"], idx)


def _candidates(L, M, rg):
    delays = np.zeros((M, L)); delays[:, 1:] = rg.uniform(-4, 9, (M, L - 1))
    return delays, rg.uniform(0.3, 3.0, (M, L)), np.exp(rg.uniform(np.log(0.3), np.log(60.0), M))


def _check_oracle(op, delays, alpha, rho, ll, grad, where):
    for m in range(len(rho)):
        rl, rgd = op.loglik_grad(delays[m], alpha[m], rho[m])
        assert abs(ll[m] - rl) <= LL_RTOL * abs(rl), (where, m, ll[m], rl)
        if grad is not None:
            assert np.max(np.abs(grad[m] - rgd)) <= GRAD_RTOL * np.max(np.abs(rgd)), (where, m, grad[m], rgd)


def _run_switched(env, code, **inputs):
    """Run `code` in a fresh interpreter with the switches in `env` (the library reads them once per process).  The code
    sees the inputs as `z` and returns arrays with out(name, array)."""
    prelude = ("import os, sys, numpy as np\nsys.path.insert(0, %r); sys.path.insert(0, %r)\nimport gpcc_b200\n"
               "tmp = sys.argv[1]\nz = np.load(os.path.join(tmp, 'in.npz'))\n"
               "def out(name, a): np.save(os.path.join(tmp, name + '.npy'), np.asarray(a))\n") % (ROOT, TESTS)
    with tempfile.TemporaryDirectory() as tmp:
        np.savez(os.path.join(tmp, "in.npz"), **inputs)
        r = subprocess.run([sys.executable, "-c", prelude + code, tmp], env=dict(os.environ, **env), capture_output=True,
                           text=True, timeout=600)
        assert r.returncode == 0, (env, r.stderr[-2500:])
        return {f[:-4]: np.load(os.path.join(tmp, f)) for f in os.listdir(tmp) if f.endswith(".npy")}


# ---- A. fused evaluator (small_eval.cuh, small_sweep.cu) ------------------------------------------------------------------
BUCKET_EDGES = (2, 7, 8, 119, 120, 151, 152, 159, 160, 199)    # first and last N of each thread count (32 ... 352 threads)


def test_every_small_size_matches_oracle(ctx):
    """N = 2 ... 199 (T = 1 ... 25 register tiles, every thread count of the fused path), 1-3 ragged bands, logL forward-only
    and with gradient against the oracle.  The forward-only elimination skips the tiles that no longer feed a pivot; the
    header of small_eval.cuh promises the same bits as the full sweep for logL, so the two modes must agree exactly."""
    for N in range(2, 200):
        rg = np.random.default_rng(N)
        nper = _split(N, max(1, min(1 + N % 3, N // 2)), rg)
        t, y, s, d = gpcc_b200.synthetic_bands(nper, seed=N, span=float(rg.uniform(8.0, 40.0)))
        delays, alpha, rho = _candidates(len(nper), 3, rg)
        for kernel in (oracle.KERNELS if N in BUCKET_EDGES else (oracle.KERNELS[N % 4],)):
            p = Problem(t, y, s, kernel, ctx)
            ll, grad, info = p.loglik_batch(delays, alpha, rho, want_grad=True)
            assert ctx.stats()["path"] == 0
            ll_f, info_f = p.loglik_batch(delays, alpha, rho)
            assert np.all(info == 0) and np.all(info_f == 0), (N, nper, kernel)
            assert np.array_equal(ll_f, ll), (N, nper, kernel, ll_f - ll)
            _check_oracle(oracle.Problem(t, y, s, kernel), delays, alpha, rho, ll, grad, (N, nper, kernel))
            p.close()


# (N, kernel, distinct candidates, seed of the light curves, seed of the candidates)
DISPATCH_CASES = [pytest.param(N, oracle.KERNELS[k % 4], 3, 40 + k, k, id=str(N))
                  for k, N in enumerate((60, 119, 120, 151, 159, 199))]
DISPATCH_CASES += [pytest.param(N, kernel, 5, N, N, id=f"{N}-{kernel}") for N, kernel in ((60, "rbf"), (151, "matern52"))]


@pytest.mark.parametrize("N,kernel,ncand,seed,cand_seed", DISPATCH_CASES)
def test_batch_size_dispatch_is_bitwise_stable(ctx, nsm, N, kernel, ncand, seed, cand_seed):
    """The batch kernel's instantiation depends on M: <128,2> / <128,3> for T <= 15, <224,1> / <192,2> for T = 16-19,
    <224,1> for T = 20, <352,1> for T >= 21.  A few distinct candidates repeated to M = 1, 3, SMs, SMs+1, 3 SMs-1 and 3 SMs:
    every copy must be bitwise the result of the M = 1 call, with and without gradient."""
    t, y, s, d = gpcc_b200.synthetic_bands(_bands(N), seed=seed, span=25.0)
    p = Problem(t, y, s, kernel, ctx)
    delays, alpha, rho = _candidates(3, ncand, np.random.default_rng(cand_seed))
    one = [p.loglik_batch(delays[j:j + 1], alpha[j:j + 1], rho[j:j + 1], want_grad=True) for j in range(ncand)]
    one_f = [p.loglik_batch(delays[j:j + 1], alpha[j:j + 1], rho[j:j + 1])[0] for j in range(ncand)]
    _check_oracle(oracle.Problem(t, y, s, kernel), delays, alpha, rho, np.array([o[0][0] for o in one]),
                  np.array([o[1][0] for o in one]), (N, kernel))
    for M in (1, 3, nsm, nsm + 1, 3 * nsm - 1, 3 * nsm):
        rep = np.arange(M) % ncand
        ll, grad, info = p.loglik_batch(delays[rep], alpha[rep], rho[rep], want_grad=True)
        ll_f, info_f = p.loglik_batch(delays[rep], alpha[rep], rho[rep])
        assert np.all(info == 0) and np.all(info_f == 0)
        for j in range(min(M, ncand)):
            sel = rep == j
            assert np.all(ll[sel] == one[j][0][0]) and np.all(grad[sel] == one[j][1][0]), (N, M, j)
            assert np.all(ll_f[sel] == one_f[j][0]), (N, M, j)


# ---- B. persistent fit kernel (small_fit.cu, lbfgs.h, nm.h) -----------------------------------------------------------------
def _screen(p, delays, theta0, rhomin, rhomax):
    """Host-side screening: logL of every start point ([P][L+1] shared or [M][P][L+1] per candidate), shape [M][P]."""
    M = len(delays)
    th = np.broadcast_to(theta0, (M,) + theta0.shape[-2:])
    return np.stack([p.loglik_theta_batch(delays, th[:, j], rhomin, rhomax)[0] for j in range(th.shape[1])], 1)


# Start points whose transforms are exact in any libm: softplus(x) = x for x >= 37 (exp(-x) is below half an ulp of x) and
# logistic(0) = 1/2, logistic(+-40) = 1 / 0, so rho = 49.95, rhomax or rhomin with or without a fused multiply-add.
EXACT_STARTS = np.array([[38.0, 40.0, 45.0, 0.0], [50.0, 39.0, 41.0, 0.0], [40.0, 40.0, 40.0, 40.0], [44.0, 38.5, 42.0, -40.0]])
# Drawn start points: the fit kernel unpacks theta with the device's exp / log1p / tanh and a fused multiply-add, the host
# reference with glibc's and separate roundings.  alpha and rho then differ in their last bits, and logL by up to 4e-13
# relative (measured on B200: N = 119, rbf and N = 199, OU), while EXACT_STARTS give the same bits on both sides.
DRAWN_RTOL = 1e-12


def _check_screening(r, scr, theta0, where, rtol=DRAWN_RTOL):
    srt = np.sort(scr, axis=1)
    assert np.all(srt[:, -1] - srt[:, -2] > 1e-10 * np.abs(srt[:, -1])), where       # the arg-max cannot flip on the last bits
    best = np.argmax(scr, axis=1)
    th = np.broadcast_to(theta0, (len(scr),) + theta0.shape[-2:])
    if rtol == 0:
        assert np.array_equal(r["loglikel"], scr.max(axis=1)), where
    else:
        assert np.all(np.abs(r["loglikel"] - scr.max(axis=1)) <= rtol * np.abs(scr.max(axis=1))), where
    assert np.array_equal(r["theta"], th[np.arange(len(scr)), best]), where
    assert np.all(r["nfev"] == scr.shape[1]) and np.all(r["info"] == 1), where


@pytest.mark.parametrize("N", [60, 119, 151, 159, 199])
def test_fit_screening_every_instantiation(ctx, nsm, N):
    """iterations = 0: the fit kernel only screens its P = 4 start points.  M = 5, SMs+1 and 3 SMs reach every
    instantiation of small_fit.cu at this N, with L-BFGS and with Nelder-Mead compiled in.  With start points whose
    transforms are exact the screening maximum is bitwise that of the batch kernel."""
    k = [60, 119, 151, 159, 199].index(N)
    kernel = oracle.KERNELS[k % 4]
    t, y, s, d = gpcc_b200.synthetic_bands(_bands(N), seed=60 + k, span=25.0)
    p = Problem(t, y, s, kernel, ctx)
    rg = np.random.default_rng(k)
    delays = np.zeros((3 * nsm, 3)); delays[:, 1:] = rg.uniform(-3, 8, (3 * nsm, 2))
    for theta0, rtol in ((gpcc_b200.initial_solutions(y, 7 + k, 1, 4, 0.1, 100.0)[0][0], DRAWN_RTOL), (EXACT_STARTS, 0)):
        scr = _screen(p, delays, theta0, 0.1, 100.0)
        for opt in ("lbfgs", "neldermead"):
            for M in (5, nsm + 1, 3 * nsm):
                r = p.fit_batch(delays[:M], theta0, iterations=0, rhomin=0.1, rhomax=100.0, optimizer=opt)
                _check_screening(r, scr[:M], theta0, (N, opt, M, rtol), rtol)


@pytest.mark.parametrize("Mkind", ["40", "3sm"])
def test_per_candidate_start_points_follow_their_candidate(ctx, nsm, Mkind):
    """theta0[M][P][L+1] with its own start points per candidate, and delay spreads that make the work-queue sort of
    fit_shard_device (largest spread first) reorder the candidates: every candidate must screen and fit from ITS start
    points, whatever queue position it gets.  A fitted candidate is bitwise the same as the fit of that candidate alone."""
    M = 40 if Mkind == "40" else 3 * nsm
    t, y, s, d = gpcc_b200.synthetic_bands([30, 30], seed=70, span=25.0)
    p = Problem(t, y, s, "matern32", ctx)
    rg = np.random.default_rng(71)
    delays = np.zeros((M, 2)); delays[:, 1] = rg.uniform(-8.0, 12.0, M)
    order = np.argsort(-np.abs(delays[:, 1]), kind="stable")
    assert not np.array_equal(order, np.arange(M))
    var_y = np.array([np.var(a, ddof=1) for a in y])
    P = 3
    theta0 = np.empty((M, P, 3))
    theta0[:, :, :2] = oracle.invmakepositive(var_y * rg.uniform(0.3, 1.7, (M, P, 2)))
    theta0[:, :, 2] = oracle.invtransformbetween(rg.uniform(0.5, 20.0, (M, P)), 0.1, 100.0)
    scr = _screen(p, delays, theta0, 0.1, 100.0)
    r0 = p.fit_batch(delays, theta0, iterations=0, rhomin=0.1, rhomax=100.0)
    _check_screening(r0, scr, theta0, M)
    r = p.fit_batch(delays, theta0, iterations=300, rhomin=0.1, rhomax=100.0)
    for c in sorted({0, 1, int(order[0]), int(order[-1]), M // 2, M - 2, M - 1}):
        one = p.fit_batch(delays[c:c + 1], theta0[c:c + 1], iterations=300, rhomin=0.1, rhomax=100.0)
        assert r["loglikel"][c] == one["loglikel"][0] and np.array_equal(r["theta"][c], one["theta"][0]), (M, c)
        assert r["nfev"][c] == one["nfev"][0], (M, c)
        assert r["loglikel"][c] >= scr[c].max() - 1e-9, (M, c)


def _grid_fit(ctx, N, M):
    """A fitted 2-band grid of M delay candidates at size N: (t, y, s), problem, delays, start points, fit result."""
    t, y, s, d = gpcc_b200.synthetic_bands(_bands(N, 2), seed=80 + N)
    p = Problem(t, y, s, "matern32", ctx)
    delays = np.stack([np.zeros(M), np.linspace(-5.0, 10.0, M)], 1)
    theta0 = gpcc_b200.initial_solutions(y, 1, 1, 5, 0.1, 300.0)[0][0]
    return (t, y, s), p, delays, theta0, p.fit_batch(delays, theta0, iterations=1000, rhomin=0.1, rhomax=300.0)


@pytest.fixture(scope="module")
def grid60(ctx, nsm):
    return _grid_fit(ctx, 60, 3 * nsm)


@pytest.mark.parametrize("N", [60, 151, 199])
def test_lbfgs_does_not_depend_on_the_instantiation(ctx, nsm, grid60, N):
    """The same L-BFGS state machine in the instantiation of a big grid (<128,3> at N = 60, <192,2> at N = 151) and of a
    20-candidate call (<128,2>, <224,1>): loglikel, theta and the evaluation count bitwise equal; three candidates against
    the oracle's L-BFGS."""
    (t, y, s), p, delays, theta0, r = grid60 if N == 60 else _grid_fit(ctx, N, nsm + 1)
    r20 = p.fit_batch(delays[:20], theta0, iterations=1000, rhomin=0.1, rhomax=300.0)
    assert np.array_equal(r["loglikel"][:20], r20["loglikel"]) and np.array_equal(r["theta"][:20], r20["theta"])
    assert np.array_equal(r["nfev"][:20], r20["nfev"])
    for m in (0, 7, 19):
        o = oracle.gpcc(t, y, s, kernel="matern32", delays=delays[m], iterations=1000, rhomin=0.1, rhomax=300.0,
                        theta0=theta0[None], optimizer="lbfgs")
        tol = 1e-5 if np.min(r["alpha"][m]) < 1e-6 else FIT_ATOL          # collapsed scale: see test_random_problems_match_oracle
        assert r["loglikel"][m] >= o[0] - tol, (N, m, r["loglikel"][m], o[0])


def test_device_fit_equals_host_loop_at_three_ctas_per_sm(grid60):
    """test_device_resident_fit_equals_host_driven_loop at N = 60 with 3 SMs candidates (the <128,3> instantiation) against
    the host-driven batched L-BFGS of GPCC_FIT_HOST=1, with that test's assertions."""
    (t, y, s), p, delays, theta0, r = grid60
    code = ("from test_gpu_dispatch import _unpack\n"
            "p = gpcc_b200.Problem(*_unpack(z), 'matern32')\n"
            "r = p.fit_batch(z['delays'], z['theta0'], iterations=1000, rhomin=0.1, rhomax=300.0)\n"
            "out('ll', r['loglikel']); out('nfev', r['nfev'])\n")
    host = _run_switched({"GPCC_FIT_HOST": "1"}, code, delays=delays, theta0=theta0, **_pack(t, y, s))
    gap = np.abs(r["loglikel"] - host["ll"])
    assert np.median(gap) < 1e-9 and np.sum(gap > 1e-6) <= len(gap) // 50, (np.median(gap), np.sum(gap > 1e-6))
    assert abs(r["nfev"].mean() - host["nfev"].mean()) < 0.05 * host["nfev"].mean()


@pytest.mark.parametrize("N", [60, 199])
def test_nelder_mead_other_kernels_match_oracle(ctx, N):
    """optimizer="neldermead" has been compared with the oracle for matern32 only: OU, rbf and matern52 here, in the <128,2>
    (N = 60) and <352,1> (N = 199) instantiations, thresholds of test_device_nelder_mead_matches_oracle_nelder_mead."""
    for k, kernel in enumerate(("OU", "rbf", "matern52")):
        t, y, s, d = gpcc_b200.synthetic_bands(_bands(N, 2), seed=90 + k, span=25.0)
        p = Problem(t, y, s, kernel, ctx)
        theta0 = gpcc_b200.initial_solutions(y, 3 + k, 1, 3, 0.1, 100.0)[0][0]
        delays = np.stack([np.zeros(4), [1.0, 2.0, 2.5, 3.5]], 1)
        r = p.fit_batch(delays, theta0, iterations=1000, rhomin=0.1, rhomax=100.0, optimizer="neldermead")
        for m in range(4):
            o = oracle.gpcc(t, y, s, kernel=kernel, delays=delays[m], iterations=1000, rhomin=0.1, rhomax=100.0,
                            theta0=theta0[None], optimizer="neldermead")
            assert abs(r["loglikel"][m] - o[0]) < 3e-5, (N, kernel, m, r["loglikel"][m], o[0])


# ---- C. tiled path (large_path.cu) ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("regime", ["wave512", "wave128", "wave32"])
def test_gradient_batch_one_past_a_full_wave(ctx, regime):
    """Gradient batches of one evaluation more than a full wave in each default wave regime (N < 1024: 512 matrices,
    N < 4096: 128, N < 8192: 32): the second wave starts at e0 > 0 in the gradient reduction and the finalisation.  Copies
    of a few distinct candidates, every copy bitwise equal to the others and to an M = 1 call; the distinct candidates
    against the oracle (N = 260, 1100) or the committed oracle fixture (N = 6144; about 6 GB of device memory)."""
    if regime == "wave32":
        g = load_golden("loglik_large")
        t, y, s, d = gpcc_b200.synthetic_bands([int(v) for v in g["n6144_nper"]], seed=int(g["n6144_seed"]))
        assert np.allclose([a.sum() for a in t], g["n6144_tsum"], rtol=1e-13)
        p = Problem(t, y, s, str(g["kernel"]), ctx)
        delays, alpha, rho = g["n6144_delays"], g["n6144_alpha"], g["n6144_rho"]
        rep = np.r_[np.zeros(17, int), np.ones(16, int)]        # the 33rd evaluation, alone in wave 2, is candidate 1
    else:
        nper, kernel, M = ([100, 90, 70], "matern32", 513) if regime == "wave512" else ([400, 380, 320], "OU", 129)
        t, y, s, d = gpcc_b200.synthetic_bands(nper, seed=5)
        p = Problem(t, y, s, kernel, ctx)
        rg = np.random.default_rng(9)
        delays = np.zeros((3, 3)); delays[:, 1:] = rg.uniform(0, 6, (3, 2))
        alpha, rho = rg.uniform(0.5, 2.5, (3, 3)), np.array([1.5, 4.0, 7.0])
        rep = np.arange(M) % 3                                  # the last evaluation (wave 2) is candidate 2
    ll, grad, info = p.loglik_batch(delays[rep], alpha[rep], rho[rep], want_grad=True)
    assert ctx.stats()["path"] == 1 and np.all(info == 0)
    for j in range(len(rho)):
        l1, g1, i1 = p.loglik_batch(delays[j:j + 1], alpha[j:j + 1], rho[j:j + 1], want_grad=True)
        sel = rep == j
        assert np.all(ll[sel] == l1[0]) and np.all(grad[sel] == g1[0]), (regime, j)
    if regime == "wave32":
        assert np.max(np.abs(ll[[0, 17]] - g["n6144_ll"]) / np.abs(g["n6144_ll"])) < LL_RTOL
        gr = g["n6144_grad"]
        assert np.max(np.abs(grad[[0, 17]] - gr) / np.max(np.abs(gr), axis=1, keepdims=True)) < GRAD_RTOL
    else:
        _check_oracle(oracle.Problem(t, y, s, kernel), delays, alpha, rho, ll[:3], grad[:3], regime)


def _sweep_inputs(L=3):
    c2, c3 = np.arange(0.0, 2.51, 0.5), np.arange(0.0, 7.01, 1.0)
    delays = np.array([[0.0, a, b] for b in c3 for a in c2])          # 48 candidates, 8 distinct last delays
    M = len(delays)
    return delays, np.tile([0.9, 1.7, 2.2], (M, 1)), np.full(M, 3.1)


def _schedule_workloads(ctx=None):
    """The three workloads of test_tiled_schedule_invariance; run in-process and under the schedule switches."""
    res = {}
    t, y, s, d = gpcc_b200.synthetic_bands([150, 130, 93], seed=12)           # N = 373
    p = Problem(t, y, s, "matern32", ctx)
    rg = np.random.default_rng(13)
    delays = np.zeros((7, 3)); delays[:, 1:] = rg.uniform(0, 5, (7, 2))
    res["ll_i"], res["grad_i"], info = p.loglik_batch(delays, rg.uniform(0.5, 2.5, (7, 3)), rg.uniform(1.0, 6.0, 7), want_grad=True)
    assert np.all(info == 0)
    t, y, s, d = gpcc_b200.synthetic_bands([256, 256, 200], seed=21)          # N = 712
    p = Problem(t, y, s, "matern52", ctx)
    res["ll_ii"], info = p.loglik_batch(*_sweep_inputs())
    res["n_tau_cache"] = np.array((ctx or gpcc_b200.default_context()).stats()["n_tau_cache"])
    assert np.all(info == 0)
    st = p.fit_state([0.0, 1.5, 3.0], [1.1, 1.8, 2.3], 2.9)
    res["postb_mu"], res["postb_S"] = st.postb()
    tt = np.linspace(-5.0, 110.0, 100)
    res["mu_iii"], res["sd_iii"], res["S_iii"], _ = st.predict([tt[:34], tt[34:67], tt[67:]], full_cov=True)
    st.close()
    return res


def test_tiled_schedule_invariance(ctx):
    """Wave size and look-ahead are schedules, not arithmetic.  Without look-ahead (one stream, no ev_panel / ev_bulk events)
    every output is bitwise the default's: a missing dependency between the two streams shows as a mismatch.  With waves
    of 1 or 3 matrices the gradient batch and the fitted state are bitwise the same; the cached sweep is equal to 1e-14,
    because another candidate leads each wave (it sums log-det and quadratic form of the shared block)."""
    ref = _schedule_workloads(ctx)
    assert ref["n_tau_cache"] == 48
    code = "from test_gpu_dispatch import _schedule_workloads\nfor k, v in _schedule_workloads().items(): out(k, v)\n"
    for env in ({"GPCC_LARGE_NO_LOOKAHEAD": "1"}, {"GPCC_LARGE_WAVE": "1"}, {"GPCC_LARGE_WAVE": "3"},
                {"GPCC_LARGE_WAVE": "3", "GPCC_LARGE_NO_LOOKAHEAD": "1"}):
        got = _run_switched(env, code)
        assert got["n_tau_cache"] == 48, env
        for k in ref:
            if k == "ll_ii" and "GPCC_LARGE_WAVE" in env:
                assert np.max(np.abs(got[k] - ref[k]) / np.abs(ref[k])) < 1e-14, (env, k)
            else:
                assert np.array_equal(got[k], ref[k]), (env, k)


def test_no_state_leaks_between_problems(ctx):
    """Two problems of the same shape (same T, Tq, Tc) share the context's workspace and last-band cache: a sweep of A,
    then of B, a fitted state of B, and A again gives A's first result bitwise."""
    pa = Problem(*gpcc_b200.synthetic_bands([256, 256, 200], seed=21)[:3], "matern52", ctx)
    pb = Problem(*gpcc_b200.synthetic_bands([256, 256, 200], seed=22)[:3], "matern52", ctx)
    a1, _ = pa.loglik_batch(*_sweep_inputs())
    b1, _ = pb.loglik_batch(*_sweep_inputs())
    assert ctx.stats()["n_tau_cache"] == 48 and not np.any(a1 == b1)
    st = pb.fit_state([0.0, 0.5, 4.0], [0.9, 1.7, 2.2], 3.1)
    st.predict([np.linspace(0, 100, 10)] * 3, full_cov=True)
    a2, _ = pa.loglik_batch(*_sweep_inputs())
    assert np.array_equal(a1, a2)
    st.close()


DESTROY_ORDERS = list(itertools.permutations(("ctx", "problem", "state")))


@pytest.mark.parametrize("order", DESTROY_ORDERS, ids=["-".join(o) for o in DESTROY_ORDERS])
def test_objects_may_be_destroyed_in_any_order(order):
    """A context, a problem and a caller's fit state may be destroyed in any order (garbage-collected hosts run finalizers
    in unspecified order, include/gpcc_b200.h), each while it holds device resources: the context a tiled-path workspace
    with a filled last-band cache, the problem the cached fitted state of postb.  Afterwards a fresh context reproduces the
    first sweep bitwise.  gpcc_fit_state_destroy used to read the problem the state was made from: in the orders that
    destroy the problem before the state, that read freed host memory, which is not guaranteed to fail, so on that code these cases
    were not guaranteed to fail either."""
    data = gpcc_b200.synthetic_bands([256, 256, 200], seed=21)[:3]          # N = 712: the tiled path
    sweep = _sweep_inputs()
    ctx = gpcc_b200.Context(1)
    p = Problem(*data, "matern52", ctx)
    ref, info = p.loglik_batch(*sweep)
    assert np.all(info == 0) and ctx.stats()["path"] == 1 and ctx.stats()["n_tau_cache"] > 0
    p.postb([0.0, 1.5, 3.0], [1.1, 1.8, 2.3], 2.9)
    objs = {"ctx": ctx, "problem": p, "state": p.fit_state([0.0, 0.5, 4.0], [0.9, 1.7, 2.2], 3.1)}
    for name in order:
        objs[name].close()
    ctx2 = gpcc_b200.Context(1)
    again, _ = Problem(*data, "matern52", ctx2).loglik_batch(*sweep)
    assert np.array_equal(again, ref)
    ctx2.close()


def test_rejected_device_id_leaves_no_cuda_error_behind():
    """A context asked for a device id outside 0 .. count-1 fails before any CUDA call uses that id.  A call with the bad
    id would leave cudaErrorInvalidDevice as the thread's last error, and the next launch check (the fused evaluator, the
    fitted state's kernels) would report it as its own failure."""
    import torch
    t, y, s, d = gpcc_b200.synthetic_bands([20, 15], seed=3, span=10.0)
    for bad in (-1, torch.cuda.device_count()):
        with pytest.raises(gpcc_b200.GpccError):
            gpcc_b200.Context(devices=[bad])
        ctx = gpcc_b200.Context(1)
        p = Problem(t, y, s, "OU", ctx)
        ll, info = p.loglik_batch([d], [[1.0, 1.2]], [2.0])
        assert info[0] == 0 and np.isfinite(ll[0]), bad
        p.postb(d, [1.0, 1.2], 2.0)
        p.close(); ctx.close()


# ---- D. fitted state (predict.cu) ---------------------------------------------------------------------------------------------
def _woodbury_reference(t, y, s, kernel, delays, alpha, rho, ttest):
    """The form predict.cu's header states, in float64 on the host: A = K + Sobs = Lc Lc' (scipy), V = Lc^-1 Q, u = Lc^-1 Y,
    Sigma_postb = (Sigma_b^-1 + V'V)^-1, mu_postb = Sigma_postb (V'u + Sigma_b^-1 mu_b), w = u - V mu_postb, Z = Lc^-1 k*,
    mu = Z'w + Q* mu_postb, Sigma = c** - Z'Z + R' Sigma_postb R + 1e-8 I with R = Q*' - V'Z."""
    op = oracle.Problem(t, y, s, kernel)
    L = op.L
    Lc = sla.cholesky(oracle.delayed_covariance(kernel, alpha, delays, rho, op.t) + np.diag(op.sobs), lower=True)
    Q = (op.band[:, None] == np.arange(L)[None, :]).astype(np.float64)
    V, u = sla.solve_triangular(Lc, Q, lower=True), sla.solve_triangular(Lc, op.Y, lower=True)
    Sp = np.linalg.inv(np.diag(1.0 / op.Sigmab) + V.T @ V)
    Sp = 0.5 * (Sp + Sp.T)
    mup = Sp @ (V.T @ u + op.mub / op.Sigmab)
    w = u - V @ mup
    tt = [np.asarray(a, dtype=np.float64) for a in ttest]
    bt = np.repeat(np.arange(L), [len(a) for a in tt])
    Z = sla.solve_triangular(Lc, oracle.delayed_covariance(kernel, alpha, delays, rho, op.t, tt), lower=True)
    R = (np.arange(L)[:, None] == bt[None, :]).astype(np.float64) - V.T @ Z
    S = oracle.delayed_covariance(kernel, alpha, delays, rho, tt) - Z.T @ Z + R.T @ Sp @ R
    S = 0.5 * (S + S.T) + 1e-8 * np.eye(len(bt))
    return Z.T @ w + mup[bt], np.sqrt(np.maximum(np.diag(S), 1e-6)), S, mup, Sp, Lc


def _gauss_logpdf(mu, S, yt):
    c = sla.cholesky(S, lower=True)
    z = sla.solve_triangular(c, yt - mu, lower=True)
    return -0.5 * (len(yt) * np.log(2.0 * np.pi) + 2.0 * np.sum(np.log(np.diag(c))) + z @ z)


def test_woodbury_reference_reproduces_exact_arithmetic():
    """The float64 reference of the predictions below, against the 50-digit values of tests/golden/pred_exact.npz."""
    g = load_golden("pred_exact")
    for tag in ("a", "b"):
        idx = np.cumsum(g[tag + "_n"])[:-1]
        t, y, s = np.split(g[tag + "_t"], idx), np.split(g[tag + "_y"], idx), np.split(g[tag + "_s"], idx)
        tt = np.split(g[tag + "_ttest"], np.cumsum(g[tag + "_ntest"])[:-1])
        mu, sd, S, mup, Sp, _ = _woodbury_reference(t, y, s, str(g[tag + "_kernel"]), g[tag + "_delays"], g[tag + "_alpha"],
                                                    float(g[tag + "_rho"]), tt)
        assert np.max(np.abs(mu - g[tag + "_pred_mu"]) / np.abs(g[tag + "_pred_mu"])) < 1e-10
        assert np.max(np.abs(sd - g[tag + "_pred_sd"]) / g[tag + "_pred_sd"]) < 1e-10
        assert np.max(np.abs(S - g[tag + "_pred_Sigma"])) / np.max(np.abs(g[tag + "_pred_Sigma"])) < 1e-10
        assert np.max(np.abs(mup - g[tag + "_postb_mu"]) / np.abs(g[tag + "_postb_mu"])) < 1e-10
        assert np.max(np.abs(Sp - g[tag + "_postb_Sigma"])) / np.max(np.abs(g[tag + "_postb_Sigma"])) < 1e-10


PRED_EDGES = [(9, 1), (63, 7), (64, 8), (65, 9), (128, 65), (129, 64), (200, 129), (455, 1030)]


def _pred_case(N, NT, L, seed):
    rg = np.random.default_rng(seed)
    nper = _bands(N, L)
    t, y, s, d = gpcc_b200.synthetic_bands(nper, seed=seed, span=max(12.0, 0.4 * N / L))
    hi = max(a.max() for a in t)
    tt = [np.sort(rg.uniform(-2.0, hi + 2.0, c)) for c in _bands(NT, L)]
    return t, y, s, tt, rg


@pytest.mark.parametrize("N,NT", PRED_EDGES + [(100, 40)], ids=[f"N{n}-NT{m}" for n, m in PRED_EDGES] + ["L8"])
def test_predictions_at_tile_edges(ctx, N, NT):
    """Fitted-state predictions where the kernels of predict.cu change tiles: 64-row trsm blocks and 8-column CTAs, 64-wide
    gemm_tn tiles, 128-wide factor tiles, more test points than the 1024 threads of chol_logpdf_kernel; and 8 bands of which
    some get no test point.  mu, sigma, the full Sigma and the test log-likelihood against the float64 Woodbury reference."""
    L = 8 if (N, NT) == (100, 40) else (2 if N < 100 else 3)
    kernel = oracle.KERNELS[(N + NT) % 4]
    t, y, s, tt, rg = _pred_case(N, NT, L, seed=N + NT)
    if L == 8:
        tt[2], tt[5] = tt[2][:0], tt[5][:0]
        NT = sum(len(a) for a in tt)
    delays, alpha, rho = np.r_[0.0, rg.uniform(0.0, 4.0, L - 1)], rg.uniform(0.7, 2.2, L), float(rg.uniform(1.0, 5.0))
    p = Problem(t, y, s, kernel, ctx)
    st = p.fit_state(delays, alpha, rho)
    mu, sd, S, _ = st.predict(tt, full_cov=True)
    rmu, rsd, rS, rmup, rSp, _ = _woodbury_reference(t, y, s, kernel, delays, alpha, rho, tt)
    assert mu.shape == (NT,) and S.shape == (NT, NT)
    assert np.max(np.abs(mu - rmu) / np.abs(rmu)) < PRED_RTOL
    assert np.max(np.abs(sd - rsd) / rsd) < PRED_RTOL
    assert np.max(np.abs(S - rS)) / np.max(np.abs(rS)) < PRED_RTOL
    mu_b, S_b = st.postb()
    assert np.max(np.abs(mu_b - rmup) / np.abs(rmup)) < PRED_RTOL and np.max(np.abs(S_b - rSp)) / np.max(np.abs(rSp)) < PRED_RTOL
    yt = [rmu_l + rg.normal(0.0, 0.5, len(a)) for rmu_l, a in zip(np.split(rmu, np.cumsum([len(a) for a in tt])[:-1]), tt)]
    st_ = [np.full(len(a), 0.3) for a in tt]
    ll, info = st.predict_loglik(tt, yt, st_)
    ref = _gauss_logpdf(rmu, rS + 0.09 * np.eye(NT), np.concatenate(yt))
    assert info == 0 and abs(ll - ref) < PRED_RTOL * abs(ref), (ll, ref)
    st.close()


@pytest.mark.parametrize("N", [129, 455])
def test_sampler_at_tile_edges(ctx, N):
    """f = Lc z for sizes that cross the 256-row CTAs of trmv_lower_kernel and its 4-sample groups."""
    t, y, s, d = gpcc_b200.synthetic_bands(_bands(N), seed=N)
    delays, alpha, rho = np.array([0.0, 1.0, 2.5]), np.array([1.0, 1.6, 0.8]), 2.2
    st = Problem(t, y, s, "matern32", ctx).fit_state(delays, alpha, rho)
    op = oracle.Problem(t, y, s, "matern32")
    Lc = np.linalg.cholesky(oracle.delayed_covariance("matern32", alpha, delays, rho, t) + np.diag(op.sobs))
    for ns in (1, 5):
        f, z = st.sample(seed=11 + ns, nsamples=ns, return_z=True)
        assert f.shape == (ns, N) and np.max(np.abs(f - z @ Lc.T)) < 1e-10 * np.max(np.abs(f)), (N, ns)
    st.close()
