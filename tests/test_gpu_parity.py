"""GPU parity tests (run with -m gpu on a B200): the CUDA path, called through the C ABI, against the oracle
and the committed golden fixtures.  Tolerances are the ones BASELINE.json's north_star states:
  fixed-hyperparameter log-likelihood   1e-10 relative
  optimised loglikel                    1e-6 absolute (vs the oracle's L-BFGS optimum; Nelder-Mead stops earlier)
  posterior delay probabilities         1e-4 absolute
  pred means / standard deviations      1e-8 relative
"""
import numpy as np
import pytest

import gpcc_b200
import oracle
from conftest import load_golden
from gpcc_b200 import Problem

pytestmark = pytest.mark.gpu

LL_RTOL = 1e-10
GRAD_RTOL = 1e-8          # gradient is not toleranced by north_star; it only steers the optimiser
FIT_ATOL = 1e-6
POST_ATOL = 1e-4
PRED_RTOL = 1e-8

GOLDEN_LL = [f"loglik_{b}_{k}" for b in ("2band", "3band") for k in ("OU", "rbf", "matern32", "matern52")] + \
            ["loglik_3x64_matern52", "loglik_ragged_OU", "loglik_single_band_rbf"]


@pytest.mark.parametrize("name", GOLDEN_LL)
def test_loglik_and_gradient_match_golden(ctx, name):
    g = load_golden(name)
    p = Problem(g["tb"], g["yb"], g["sb"], g["kernel"], ctx)
    assert np.allclose(p.mub, g["mub"], rtol=1e-14) and np.allclose(p.Sigmab, g["Sigmab"], rtol=1e-13)
    ll, grad, info = p.loglik_batch(g["delays"], g["alpha"], g["rho"], want_grad=True)
    assert np.all(info == 0)
    assert np.max(np.abs(ll - g["loglik"]) / np.abs(g["loglik"])) < LL_RTOL
    scale = np.max(np.abs(g["grad"]), axis=1, keepdims=True)
    assert np.max(np.abs(grad - g["grad"]) / scale) < GRAD_RTOL
    ll2, info2 = p.loglik_batch(g["delays"], g["alpha"], g["rho"])            # without gradient: identical values
    assert np.array_equal(ll2, ll)


def test_loglik_matches_oracle_on_fresh_inputs(ctx):
    t, y, s, d = oracle.simulatedata(sigma=0.5, seed=7)[:4]
    for kernel in oracle.KERNELS:
        op, p = oracle.Problem(t, y, s, kernel), Problem(t, y, s, kernel, ctx)
        rg = np.random.default_rng(3)
        M = 40
        delays = np.zeros((M, 3)); delays[:, 1:] = rg.uniform(-5, 25, (M, 2))
        alpha, rho = rg.uniform(0.05, 5.0, (M, 3)), np.exp(rg.uniform(np.log(0.1), np.log(300.0), M))
        ll, grad, info = p.loglik_batch(delays, alpha, rho, want_grad=True)
        ref = [op.loglik_grad(delays[m], alpha[m], rho[m]) for m in range(M)]
        rl, rgd = np.array([r[0] for r in ref]), np.array([r[1] for r in ref])
        assert np.all(info == 0)
        assert np.max(np.abs(ll - rl) / np.abs(rl)) < LL_RTOL, kernel
        assert np.max(np.abs(grad - rgd) / np.max(np.abs(rgd), axis=1, keepdims=True)) < GRAD_RTOL, kernel


def test_theta_space_gradient_chain_rule(ctx):
    g = load_golden("loglik_3band_matern32")
    op, p = oracle.Problem(g["tb"], g["yb"], g["sb"], "matern32"), Problem(g["tb"], g["yb"], g["sb"], "matern32", ctx)
    rg = np.random.default_rng(5)
    theta = rg.normal(0.0, 1.5, (16, 4))
    delays = np.tile([0.0, 2.0, 4.0], (16, 1))
    ll, grad, info = p.loglik_theta_batch(delays, theta, 0.1, 300.0, want_grad=True)
    for m in range(16):
        rl, rgd = op.objective_grad_theta(theta[m], delays[m], 0.1, 300.0)
        assert abs(ll[m] - rl) / abs(rl) < LL_RTOL
        assert np.max(np.abs(grad[m] - rgd)) / np.max(np.abs(rgd)) < GRAD_RTOL


def test_determinism_and_batch_independence(ctx):
    g = load_golden("loglik_3band_OU")
    p = Problem(g["tb"], g["yb"], g["sb"], "OU", ctx)
    a = p.loglik_batch(g["delays"], g["alpha"], g["rho"], want_grad=True)
    b = p.loglik_batch(g["delays"], g["alpha"], g["rho"], want_grad=True)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])             # bitwise reproducible
    perm = np.random.default_rng(0).permutation(len(g["rho"]))
    c = p.loglik_batch(g["delays"][perm], g["alpha"][perm], g["rho"][perm], want_grad=True)
    assert np.array_equal(c[0], a[0][perm]) and np.array_equal(c[1], a[1][perm])
    big = p.loglik_batch(np.tile(g["delays"], (50, 1)), np.tile(g["alpha"], (50, 1)), np.tile(g["rho"], 50))
    assert np.array_equal(big[0], np.tile(a[0], 50))                             # 1200 CTAs, several waves


def test_not_positive_definite_and_invalid_hyperparameters(ctx):
    # duplicated time stamps with zero noise: K + Sobs + B is singular -> LAPACK-style info > 0, loglik = -Inf
    t = [np.array([1.0, 1.0, 2.0, 3.0]), np.array([1.5, 2.5, 2.5])]
    y = [np.array([1.0, 2.0, 1.5, 0.5]), np.array([3.0, 2.0, 2.5])]
    s = [np.zeros(4), np.zeros(3)]
    p = Problem(t, y, s, "rbf", ctx)
    ll, grad, info = p.loglik_batch([[0.0, 0.0]], [[1.0, 1.0]], [1.0], want_grad=True)
    assert info[0] > 0 and ll[0] == -np.inf and np.all(grad == 0.0)
    # scale <= 0 / rho <= 0 are errors in delayedCovariance.jl:3-7 -> info -1, -Inf, nothing sent to the device
    ll, info = p.loglik_batch([[0.0, 0.0]] * 3, [[1.0, -1.0], [1.0, 1.0], [np.nan, 1.0]], [1.0, 0.0, 1.0])
    assert np.all(info == -1) and np.all(ll == -np.inf)
    with pytest.raises(gpcc_b200.GpccError):
        Problem([np.array([1.0])], [np.array([1.0])], [np.array([0.1])], "OU", ctx)    # var of one point is undefined
    with pytest.raises(gpcc_b200.GpccError):
        Problem(t, y, s, "cosine", ctx)


def test_empty_batch_and_single_candidate(ctx):
    g = load_golden("loglik_2band_rbf")
    p = Problem(g["tb"], g["yb"], g["sb"], "rbf", ctx)
    ll, info = p.loglik_batch(np.zeros((0, 2)), np.zeros((0, 2)), np.zeros(0))
    assert ll.shape == (0,)
    ll, info = p.loglik_batch(g["delays"][:1], g["alpha"][:1], g["rho"][:1])
    assert abs(ll[0] - g["loglik"][0]) / abs(g["loglik"][0]) < LL_RTOL


# ---- fit, posterior (configs 1-3) -------------------------------------------------------------------------
def test_cfg1_single_fit_matches_oracle(ctx, capsys):
    g = load_golden("fit_cfg1_cfg2")
    loglikel, pred, (alpha, postb, rho) = gpcc_b200.gpcc(g["tb"], g["yb"], g["sb"], kernel=gpcc_b200.matern32,
                                                        delays=g["truedelays"], iterations=1000, rhomax=300,
                                                        theta0=g["theta0"], ctx=ctx)
    out = capsys.readouterr().out
    assert "Running with random seed 1" in out and "Overall minimum is" in out        # util.jl:1-11, :228
    assert abs(loglikel - float(g["loglikel"])) < FIT_ATOL
    assert loglikel >= float(g["loglikel_nm"]) - FIT_ATOL          # never worse than the reference's Nelder-Mead
    assert np.allclose(alpha, g["alpha"], rtol=1e-4) and rho == pytest.approx(float(g["rho"]), rel=1e-4)
    # postb (:248-252) evaluated at the oracle's optimum so that only the linear algebra is compared
    p = Problem(g["tb"], g["yb"], g["sb"], "matern32", ctx)
    mu, S = p.postb(g["truedelays"], g["alpha"], float(g["rho"]))
    assert np.allclose(mu, g["postb_mu"], rtol=PRED_RTOL) and np.allclose(S, g["postb_Sigma"], rtol=PRED_RTOL)
    assert np.array_equal(S, S.T) and isinstance(postb, gpcc_b200.MvNormal)
    # pred(t::Vector) (:293-307)
    m_, sd_, _, _ = p.predict(g["truedelays"], g["alpha"], float(g["rho"]), [g["ttest"]] * 2)
    nt = len(g["ttest"])
    assert np.max(np.abs(m_.reshape(2, nt) - g["pred_mu"]) / np.abs(g["pred_mu"])) < PRED_RTOL
    assert np.max(np.abs(sd_.reshape(2, nt) - g["pred_sd"]) / g["pred_sd"]) < PRED_RTOL
    mu_b, sd_b = pred(g["ttest"])
    assert len(mu_b) == 2 and mu_b[0].shape == (nt,) and np.allclose(mu_b[1], g["pred_mu"][1], rtol=1e-4)
    # pred(t::Vector{Vector}) -> (mu, Sigma) (:259-289), ragged test sets
    mf, _, Sf, _ = p.predict(g["truedelays"], g["alpha"], float(g["rho"]), [g["ttest"][:7], g["ttest"][5:9]], full_cov=True)
    assert np.max(np.abs(mf - g["predfull_mu"]) / np.abs(g["predfull_mu"])) < PRED_RTOL
    assert np.max(np.abs(Sf - g["predfull_Sigma"])) / np.max(np.abs(g["predfull_Sigma"])) < PRED_RTOL
    assert np.array_equal(Sf, Sf.T)
    # pred(ttest, ytest, sigmatest) (:311-343), the README's numbers
    tl, info = p.predict_loglik(g["truedelays"], g["alpha"], float(g["rho"]), [[9.0, 10.0, 11.0], [9.0, 10.0, 11.0]],
                                [[6.34, 5.49, 5.38], [13.08, 12.37, 15.69]], [[0.34, 0.42, 0.2], [0.87, 0.8, 0.66]])
    assert info == 0 and abs(tl - float(g["test_loglik"])) / abs(float(g["test_loglik"])) < PRED_RTOL


def test_test_likelihood_with_duplicated_test_times(ctx):
    """pred(ttest, ytest, sigmatest) with a duplicated test time and zero test noise: only the 1e-8 jitter (:279) keeps the
    predictive covariance positive definite; device and oracle must agree on this badly conditioned case as well."""
    g = load_golden("fit_cfg1_cfg2")
    tt = [np.array([3.0, 3.0, 9.0]), np.array([4.0, 12.0])]
    yt = [np.array([6.1, 6.1, 5.5]), np.array([14.0, 13.0])]
    st = [np.zeros(3), np.array([0.5, 0.5])]
    p = Problem(g["tb"], g["yb"], g["sb"], "matern32", ctx)
    got, info = p.predict_loglik(g["truedelays"], g["alpha"], float(g["rho"]), tt, yt, st)
    ref = oracle.Problem(g["tb"], g["yb"], g["sb"], "matern32").predict_loglik(g["truedelays"], g["alpha"], float(g["rho"]), tt, yt, st)
    assert info == 0 and np.isfinite(got) and abs(got - ref) / abs(ref) < 1e-4      # cond ~ 1e10: agreement to ~1e-6 is all FP64 gives


def test_cross_validation_driver_matches_oracle(ctx):
    """performcv (src/UNUSED/performcv.jl:41-139, SURVEY 8f): fold-wise fit + held-out test log-likelihood, same folds and
    start points on both sides."""
    import io
    t, y, s, d = gpcc_b200.simulatetwolightcurves()
    folds = gpcc_b200.cv_folds([len(a) for a in t], 3, 1)
    th = []
    for k in range(3):
        ytr = [np.asarray(a)[np.asarray(f) != k] for a, f in zip(y, folds)]
        th.append(gpcc_b200.initial_solutions(ytr, 1, 1, 3, 0.1, 20.0)[0])
    got = gpcc_b200.performcv(t, y, s, delays=d, kernel=gpcc_b200.matern32, iterations=500, numberoffolds=3, folds=folds,
                              theta0=th, ctx=ctx, out=io.StringIO())
    ref = oracle.performcv(t, y, s, delays=d, kernel="matern32", iterations=500, numberoffolds=3, folds=folds, theta0=th)
    assert got.shape == (3,) and np.all(np.isfinite(got))
    assert np.max(np.abs(got - ref)) < 1e-5 * np.max(np.abs(ref))      # two optimisers, same optimum: test logL to ~1e-6


def test_cfg2_grid_posterior_matches_oracle(ctx):
    g = load_golden("fit_cfg1_cfg2")
    p = Problem(g["tb"], g["yb"], g["sb"], "matern32", ctx)
    delays = np.stack([np.zeros_like(g["cands"]), g["cands"]], 1)
    res = p.grid_posterior(delays, g["theta0"], iterations=1000, rhomin=0.1, rhomax=300.0)
    gap = np.abs(res["loglikel"] - g["ll_grid"])
    carries_mass = g["post_flat"] > 1e-12
    # same basin wherever the candidate carries posterior mass (SURVEY.md section 7 "hard parts")
    assert np.max(gap[carries_mass]) < FIT_ATOL, (np.max(gap), np.argmax(gap))
    assert np.sum(gap > FIT_ATOL) <= 2, "basin mismatches: %d" % np.sum(gap > FIT_ATOL)
    assert np.all(res["loglikel"] >= g["ll_grid_nm"] - 1e-5)      # at least as good as the reference optimiser everywhere
    assert np.max(np.abs(res["posterior"] - g["post_flat"])) < POST_ATOL
    assert np.max(np.abs(res["posterior"] - oracle.getprobabilities(g["ll_grid_nm"]))) < POST_ATOL
    assert res["posterior"].sum() == pytest.approx(1.0, abs=1e-12)
    prior = gpcc_b200.uniformpriordelay(L=1e44, z=0.0)
    res2 = p.grid_posterior(delays, g["theta0"], iterations=1000, rhomin=0.1, rhomax=300.0, logprior=prior.logpdf(g["cands"]))
    assert np.max(np.abs(res2["posterior"] - g["post_prior"])) < POST_ATOL
    # getprobabilities on the device, shape preserving, -Inf -> 0 (getprobabilities.jl:1-20)
    ll2 = g["ll_grid"][:100].reshape(10, 10).copy()
    ll2[3, 4] = -np.inf
    pp = gpcc_b200.getprobabilities(ll2, ctx=ctx)
    assert pp.shape == (10, 10) and pp[3, 4] == 0.0 and np.allclose(pp, oracle.getprobabilities(ll2), rtol=1e-12, atol=1e-300)


def test_cfg3_subgrid_three_bands(ctx):
    g = load_golden("fit_cfg3_subgrid")
    p = Problem(g["tb"], g["yb"], g["sb"], "matern32", ctx)
    res = p.grid_posterior(g["delays"], g["theta0"], iterations=1000, rhomin=0.1, rhomax=300.0)
    gap = np.abs(res["loglikel"] - g["ll"])
    assert np.max(gap[g["post"] > 1e-12]) < FIT_ATOL
    assert np.max(np.abs(res["posterior"] - g["post"])) < POST_ATOL
    assert np.allclose(g["delays"][np.argmax(res["posterior"])], [0.0, 2.0, 4.0])
    # basin report: candidates whose optimum differs from the oracle's L-BFGS by more than 1e-6 carry no mass
    assert np.all(g["post"][gap > FIT_ATOL] < 1e-12)


def test_full_size_cfg3_grid_properties(ctx):
    """BASELINE config 3 at full size (101 x 101 = 10 201 candidates): size-independent properties."""
    t, y, s, d = oracle.simulatethreelightcurves()
    p = Problem(t, y, s, "matern32", ctx)
    c = np.arange(0.0, 20.0001, 0.2)
    delays = np.array([[0.0, a, b] for b in c for a in c])            # d1 fastest (README.md:231-235)
    theta0 = gpcc_b200.initial_solutions(y, 1, 1, 5, 0.1, 300.0)[0][0]
    res = p.grid_posterior(delays, theta0, iterations=1000, rhomin=0.1, rhomax=300.0)
    post = res["posterior"].reshape(101, 101, order="F")             # reshape(posterior, n, n) in Julia
    assert post.sum() == pytest.approx(1.0, abs=1e-10) and np.all(post >= 0)
    i, j = np.unravel_index(np.argmax(post), post.shape)
    assert abs(c[i] - 2.0) <= 0.4 and abs(c[j] - 4.0) <= 0.4          # truth (2, 4)
    # the optimum can only improve on the best screening point, and re-evaluating theta-hat reproduces loglikel
    ll_chk, _ = p.loglik_batch(delays[::97], res["alpha"][::97], res["rho"][::97])
    assert np.allclose(ll_chk, res["loglikel"][::97], rtol=1e-12)
    scr = np.max(np.stack([p.loglik_theta_batch(delays[::97], np.tile(th, (len(delays[::97]), 1)), 0.1, 300.0)[0]
                           for th in theta0]), axis=0)
    assert np.all(res["loglikel"][::97] >= scr - 1e-9)
    assert np.all(res["info"] >= 0)
    # ... and against the oracle's L-BFGS optimum of ALL 10 201 candidates (tests/golden/fit_cfg3_full.npz)
    g = load_golden("fit_cfg3_full")
    assert np.array_equal(g["delays"], delays) and np.allclose(g["theta0"], theta0, rtol=0, atol=0)
    gap = np.abs(res["loglikel"] - g["ll"])
    mass = g["post"] > 1e-12
    worse = res["loglikel"] < g["ll"] - FIT_ATOL
    print("cfg3 full grid: %d candidates carry mass > 1e-12, max gap there %.2e; basin mismatches elsewhere: %d (device better on %d, "
          "oracle better on %d)" % (mass.sum(), gap[mass].max(), np.sum(gap > FIT_ATOL), np.sum(gap > FIT_ATOL) - worse.sum(), worse.sum()))
    assert np.max(gap[mass]) < FIT_ATOL
    assert np.max(np.abs(res["posterior"] - g["post"])) < POST_ATOL
    assert np.all(g["post"][gap > FIT_ATOL] < 1e-12)


def test_restarts_and_per_candidate_starts(ctx):
    g = load_golden("fit_cfg1_cfg2")
    p = Problem(g["tb"], g["yb"], g["sb"], "matern32", ctx)
    th, _ = gpcc_b200.initial_solutions(g["yb"], seed=3, numberofrestarts=3, initialrandom=4, rhomin=0.1, rhomax=300.0)
    res = p.fit_batch(np.tile(g["truedelays"], (3, 1)), th, iterations=1000, rhomin=0.1, rhomax=300.0)   # [M][P][L+1]
    assert np.max(res["loglikel"]) >= float(g["loglikel"]) - 1e-6
    ll, _, _ = gpcc_b200.gpcc(g["tb"], g["yb"], g["sb"], kernel="matern32", delays=g["truedelays"], iterations=1000,
                              rhomax=300, seed=3, numberofrestarts=3, initialrandom=4, ctx=ctx, verbose=False)
    assert ll == pytest.approx(np.max(res["loglikel"]), abs=1e-9)
    capped = p.fit_batch(g["truedelays"][None], g["theta0"], iterations=2, rhomin=0.1, rhomax=300.0)
    assert capped["info"][0] == 1 and capped["iters"][0] == 2 and capped["loglikel"][0] < float(g["loglikel"])


# ---- the reference's own optimiser on the device (nm.h): basin-for-basin comparison ---------------------------------------
def test_device_nelder_mead_matches_oracle_nelder_mead(ctx):
    """optimizer="neldermead": Optim's adaptive Nelder-Mead (:205-211) as a device state machine on forward-only evaluations,
    against the oracle's restatement of the same algorithm from the same start points.  NM stops when the simplex spread is
    below g_tol = 1e-6, so two runs whose comparisons flip on the last bits end up to ~1e-5 apart."""
    g = load_golden("fit_cfg1_cfg2")
    p = Problem(g["tb"], g["yb"], g["sb"], "matern32", ctx)
    delays = np.stack([np.zeros_like(g["cands"]), g["cands"]], 1)
    r = p.grid_posterior(delays, g["theta0"], iterations=1000, rhomin=0.1, rhomax=300.0, optimizer="neldermead")
    gap = np.abs(r["loglikel"] - g["ll_grid_nm"])
    print("cfg2 device NM vs oracle NM: median gap %.1e, max %.1e, beyond 1e-4: %d of %d; mean evaluations %.0f"
          % (np.median(gap), gap.max(), np.sum(gap > 1e-4), len(gap), r["nfev"].mean()))
    assert np.median(gap) < 1e-6 and np.max(gap[g["post_flat"] > 1e-12]) < 3e-5
    assert np.max(np.abs(r["posterior"] - oracle.getprobabilities(g["ll_grid_nm"]))) < POST_ATOL
    assert np.max(np.abs(r["posterior"] - g["post_flat"])) < POST_ATOL                 # and the same posterior as the L-BFGS fit
    ll, _, _ = gpcc_b200.gpcc(g["tb"], g["yb"], g["sb"], kernel="matern32", delays=g["truedelays"], iterations=1000, rhomax=300,
                              theta0=g["theta0"], ctx=ctx, verbose=False, optimizer="neldermead")
    assert abs(ll - float(g["loglikel_nm"])) < 3e-5 and ll <= float(g["loglikel"]) + 1e-9
    capped = p.fit_batch(delays[:4], g["theta0"], iterations=3, rhomin=0.1, rhomax=300.0, optimizer="neldermead")
    assert np.all(capped["info"] == 1) and np.all(capped["iters"] == 3)
    big = Problem(*gpcc_b200.synthetic_bands([120, 110], seed=9)[:3], "matern32", ctx)
    with pytest.raises(gpcc_b200.GpccError):                                             # tiled path: L-BFGS only
        big.fit_batch([[0.0, 1.0]], g["theta0"], iterations=10, rhomin=0.1, rhomax=300.0, optimizer="neldermead")


def test_device_nelder_mead_full_cfg3_grid_against_oracle(ctx):
    """All 10 201 candidates of BASELINE config 3 with the reference's optimiser on both sides
    (tests/golden/fit_cfg3_full_nm.npz: the oracle's Nelder-Mead, 16 CPU-minutes; here ~1.5 s)."""
    g = load_golden("fit_cfg3_full_nm")
    t, y, s, d = oracle.simulatethreelightcurves()
    p = Problem(t, y, s, "matern32", ctx)
    r = p.grid_posterior(g["delays"], g["theta0"], iterations=1000, rhomin=0.1, rhomax=300.0, optimizer="neldermead")
    gap = np.abs(r["loglikel"] - g["ll"])
    mass = g["post"] > 1e-12
    print("cfg3 full grid, NM vs NM: %d candidates with mass, max gap there %.1e; same basin (gap < 1e-4) on %d of %d candidates; "
          "mean evaluations %.0f (oracle %.0f)" % (mass.sum(), gap[mass].max(), np.sum(gap < 1e-4), len(gap), r["nfev"].mean(), g["nfev"].mean()))
    assert np.max(gap[mass]) < 3e-5
    assert np.max(np.abs(r["posterior"] - g["post"])) < POST_ATOL
    assert np.mean(gap < 1e-4) > 0.9                    # basin for basin: the two Nelder-Mead runs agree on (nearly) every candidate
    assert abs(r["nfev"].mean() - g["nfev"].mean()) < 0.1 * g["nfev"].mean()


# ---- large-N path (tile layout in HBM, DMMA trailing updates), BASELINE configs 4/5 --------------------------
@pytest.mark.parametrize("nper,kernel", [([100, 90, 70], "matern32"), ([256, 256, 256], "matern52"), ([300, 212], "OU"),
                                         ([201], "rbf"), ([64, 64, 64, 64], "matern32")])
def test_large_path_matches_oracle(ctx, nper, kernel):
    t, y, s, d = gpcc_b200.synthetic_bands(nper, seed=3)
    op, p = oracle.Problem(t, y, s, kernel), Problem(t, y, s, kernel, ctx)
    L, M = len(nper), 3
    rg = np.random.default_rng(1)
    delays = np.zeros((M, L)); delays[:, 1:] = rg.uniform(0, 6, (M, L - 1))
    alpha, rho = rg.uniform(0.5, 2.5, (M, L)), rg.uniform(1.0, 8.0, M)
    ll, grad, info = p.loglik_batch(delays, alpha, rho, want_grad=True)        # symmetric sweep (inverse + gradient)
    assert ctx.stats()["path"] == 1 and np.all(info == 0)
    ll_fwd, info_fwd = p.loglik_batch(delays, alpha, rho)                      # forward only = blocked Cholesky
    ref = [op.loglik_grad(delays[m], alpha[m], rho[m]) for m in range(M)]
    rl, rgd = np.array([r[0] for r in ref]), np.array([r[1] for r in ref])
    assert np.max(np.abs(ll - rl) / np.abs(rl)) < LL_RTOL and np.max(np.abs(ll_fwd - rl) / np.abs(rl)) < LL_RTOL
    assert np.max(np.abs(grad - rgd) / np.max(np.abs(rgd), axis=1, keepdims=True)) < GRAD_RTOL
    again = p.loglik_batch(delays, alpha, rho, want_grad=True)
    assert np.array_equal(again[0], ll) and np.array_equal(again[1], grad)      # deterministic


@pytest.mark.parametrize("nper", [[256, 256, 200], [300, 280, 330], [200, 150, 180, 220]])   # boundaries on / off the 128-wide tile boundaries; four bands
def test_last_band_cache(ctx, nper):
    """Fixed-theta sweep over three bands: what the band-1 pivots do to the rows of band 3
    depends on tau_3 alone (block (3,1) of the covariance: src/delayedCovariance.jl:23-31), so it is computed once per distinct
    tau_3 and imported by every candidate (large_path.cu, last-band cache).  Same kernels on the same operands in the same
    order: the log-likelihoods are BITWISE those of a run without the cache; oracle parity as everywhere."""
    import os, subprocess, sys, tempfile
    t, y, s, d = gpcc_b200.synthetic_bands(nper, seed=21)                              # N = 712: T = 6 tiles, Tq = 2, Tc = 4 / N = 910: T = 8, 2, 5
    p = Problem(t, y, s, "matern52", ctx)
    c2, c3 = np.arange(0.0, 2.51, 0.5), np.arange(0.0, 7.01, 1.0)
    L = len(nper)
    mk = lambda a, b: [0.0] + [1.3] * (L - 3) + [a, b]                                 # the grid runs over the last two delays
    a0 = np.array([0.9, 1.7, 2.2, 1.4])[:L]
    delays = np.array([mk(a, b) for b in c3 for a in c2])                             # 48 candidates, 8 distinct last delays
    M = len(delays)
    alpha, rho = np.tile(a0, (M, 1)), np.full(M, 3.1)
    ll, info = p.loglik_batch(delays, alpha, rho)
    st = ctx.stats()
    assert st["path"] == 1 and np.all(info == 0) and st["n_tau_cache"] == M and st["n_shared_prefix"] > 0
    op = oracle.Problem(t, y, s, "matern52")
    for m in (0, 5, 29, M - 1):
        assert abs(ll[m] - op.loglik(delays[m], alpha[m], rho[m])) / abs(ll[m]) < LL_RTOL
    code = ("import numpy as np, sys; sys.path.insert(0, %r)\nimport gpcc_b200\n"
            "t, y, s, d = gpcc_b200.synthetic_bands(%r, seed=21)\n"
            "p = gpcc_b200.Problem(t, y, s, 'matern52')\n"
            "z = np.load(sys.argv[1]); ll, info = p.loglik_batch(z['delays'], z['alpha'], z['rho'])\n"
            "assert gpcc_b200.default_context().stats()['n_tau_cache'] == 0\n"
            "np.save(sys.argv[2], ll)\n") % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))), nper)
    with tempfile.TemporaryDirectory() as tmp:
        np.savez(os.path.join(tmp, "in.npz"), delays=delays, alpha=alpha, rho=rho)
        r = subprocess.run([sys.executable, "-c", code, os.path.join(tmp, "in.npz"), os.path.join(tmp, "out.npy")],
                           env=dict(os.environ, GPCC_LARGE_NO_TAUCACHE="1"), capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr[-2000:]
        ll_plain = np.load(os.path.join(tmp, "out.npy"))
    assert np.array_equal(ll, ll_plain)
    for _ in range(3):                                                                 # deterministic (no race between the waves)
        assert np.array_equal(p.loglik_batch(delays, alpha, rho)[0], ll)
    perm = np.random.default_rng(5).permutation(M)                                     # any order of the candidates: another
    ll_p, _ = p.loglik_batch(delays[perm], alpha[perm], rho[perm])                     # candidate leads each wave (it sums
    assert np.max(np.abs(ll_p - ll[perm]) / np.abs(ll)) < 1e-14                        # log-det and quadratic form in one go)
    # mixed hyper-parameters: no cache, same numbers for the untouched candidates
    alpha2 = alpha.copy(); alpha2[7, 1] = 1.9
    ll2, _ = p.loglik_batch(delays, alpha2, rho)
    assert ctx.stats()["n_tau_cache"] == 0 and np.max(np.abs(np.delete(ll2, 7) - np.delete(ll, 7)) / np.abs(np.delete(ll, 7))) < 1e-14
    # many tau_2, few tau_3: the runs with a common tau_2 are too short to share their leading block (every matrix factorises
    # its own bands 1-2), the last-band cache serves them all the same
    c2b = np.arange(0.0, 3.76, 0.25)
    delays_b = np.array([mk(a, b) for a in c2b for b in c3[:3]])
    Mb = len(delays_b)
    ll_b, info_b = p.loglik_batch(delays_b, np.tile(alpha[0], (Mb, 1)), np.full(Mb, rho[0]))
    st_b = ctx.stats()
    assert np.all(info_b == 0) and st_b["n_tau_cache"] == Mb and st_b["n_shared_prefix"] == 0
    for m in range(Mb):
        hit = np.where(np.all(delays == delays_b[m], axis=1))[0]
        if len(hit):
            assert abs(ll_b[m] - ll[hit[0]]) / abs(ll_b[m]) < 1e-14
    assert abs(ll_b[4] - op.loglik(delays_b[4], alpha[0], rho[0])) / abs(ll_b[4]) < LL_RTOL
    # a second sweep with other hyper-parameters refills the cache (entries belong to one call)
    ll3, _ = p.loglik_batch(delays, alpha * 1.25, rho * 0.8)
    assert abs(ll3[11] - op.loglik(delays[11], alpha[11] * 1.25, rho[11] * 0.8)) / abs(ll3[11]) < LL_RTOL
    # the grid driver with iterations = 0 takes the same route
    th = np.concatenate([np.log(np.expm1(a0)), [np.log((3.1 - 0.1) / (300.0 - 3.1))]])[None]
    r = p.grid_posterior(delays, th, iterations=0, rhomin=0.1, rhomax=300.0)
    assert ctx.stats()["n_tau_cache"] == M and abs(r["posterior"].sum() - 1.0) < 1e-12


def test_structure_reuse_across_the_grid(ctx):
    """Fixed-theta sweep on the tiled path (SURVEY 8f item 2): candidates that share the hyper-parameters and the delays of all
    bands but the last share the leading block of the covariance (src/delayedCovariance.jl:23-31); a wave factorises it once.
    Same numbers as without sharing (to rounding: only the summation order of log-det / quadratic form differs), for any
    order of the candidates, ragged bands, and through the iterations=0 grid driver."""
    import os, subprocess, sys
    t, y, s, d = gpcc_b200.synthetic_bands([150, 130, 93], seed=12)                 # band boundaries not on tile boundaries
    p = Problem(t, y, s, "matern32", ctx)
    c2, c3 = np.arange(0.0, 3.01, 0.5), np.arange(0.0, 6.01, 0.25)
    delays = np.array([[0.0, a, b] for b in c3 for a in c2])                          # d1 fastest: the shared prefix is scattered
    M = len(delays)
    alpha, rho = np.tile([1.1, 1.9, 2.4], (M, 1)), np.full(M, 2.7)
    ll, info = p.loglik_batch(delays, alpha, rho)
    st = ctx.stats()
    assert st["path"] == 1 and np.all(info == 0)
    assert st["n_shared_prefix"] >= M - 2 * len(c2)                                    # all but one evaluation per wave reuse the block
    op = oracle.Problem(t, y, s, "matern32")
    for m in (0, 17, M - 1):
        assert abs(ll[m] - op.loglik(delays[m], alpha[m], rho[m])) / abs(ll[m]) < LL_RTOL
    code = ("import numpy as np, sys; sys.path.insert(0, %r)\nimport gpcc_b200\n"
            "t, y, s, d = gpcc_b200.synthetic_bands([150, 130, 93], seed=12)\n"
            "p = gpcc_b200.Problem(t, y, s, 'matern32')\n"
            "z = np.load(sys.argv[1]); ll, info = p.loglik_batch(z['delays'], z['alpha'], z['rho'])\n"
            "assert gpcc_b200.default_context().stats()['n_shared_prefix'] == 0\n"
            "np.save(sys.argv[2], ll)\n") % os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    import tempfile
    with tempfile.TemporaryDirectory() as tmp:
        np.savez(os.path.join(tmp, "in.npz"), delays=delays, alpha=alpha, rho=rho)
        r = subprocess.run([sys.executable, "-c", code, os.path.join(tmp, "in.npz"), os.path.join(tmp, "out.npy")],
                           env=dict(os.environ, GPCC_LARGE_NO_SHARE="1"), capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr[-2000:]
        ll_plain = np.load(os.path.join(tmp, "out.npy"))
    assert np.max(np.abs(ll - ll_plain) / np.abs(ll_plain)) < 1e-13
    perm = np.random.default_rng(3).permutation(M)
    ll_p, _ = p.loglik_batch(delays[perm], alpha[perm], rho[perm])
    assert np.array_equal(ll_p, ll[perm])                                              # the internal ordering does not leak out
    # mixed hyper-parameters: only equal (alpha, rho, prefix) may share
    alpha2 = alpha.copy(); alpha2[::3, 0] = 1.3
    ll2, _ = p.loglik_batch(delays, alpha2, rho)
    for m in (0, 1, 2, 3):
        assert abs(ll2[m] - op.loglik(delays[m], alpha2[m], rho[m])) / abs(ll2[m]) < LL_RTOL
    # the grid driver with iterations = 0 (the north-star fixed-theta posterior) goes through the same reuse
    th = np.concatenate([np.log(np.expm1(np.array([1.1, 1.9, 2.4]))), [np.log((2.7 - 0.1) / (300.0 - 2.7))]])[None]
    r = p.grid_posterior(delays, th, iterations=0, rhomin=0.1, rhomax=300.0)
    assert ctx.stats()["n_shared_prefix"] > 0 and abs(r["posterior"].sum() - 1.0) < 1e-12
    a_, r_ = r["alpha"][0], r["rho"][0]
    ll3, _ = p.loglik_batch(delays, np.tile(a_, (M, 1)), np.full(M, r_))
    assert np.allclose(r["loglikel"], ll3, rtol=1e-13)
    # a matrix that is not positive definite inside the shared block is reported for every candidate of the wave
    t2 = [a.copy() for a in t]; t2[0][5] = t2[0][4]
    pb = Problem(t2, y, [np.zeros_like(a) for a in s], "rbf", ctx)
    llb, infob = pb.loglik_batch(delays[:14], alpha[:14], np.full(14, 0.05))
    assert np.all(llb == -np.inf) and np.all(infob > 0) and np.all(infob <= 150)


def test_device_sampler_and_simulator(ctx):
    """gpcc_fit_state_sample: f = Lc z with Lc the cached factor of K + Sobs and z from the device's Philox / Box-Muller
    generator (the draw of src/simulatedata.jl:128-145).  Exactness through the returned deviates, distribution through
    moments, reproducibility through the seed; then the simulator built around it, fitted back."""
    t, y, s, d = gpcc_b200.synthetic_bands([90, 80, 70], seed=8)
    p = Problem(t, y, s, "OU", ctx)
    alpha, rho = np.array([1.0, 1.5, 2.0]), 3.5
    st = p.fit_state(d, alpha, rho)
    f, z = st.sample(seed=123, nsamples=3, return_z=True)
    op = oracle.Problem(t, y, s, "OU")
    K = oracle.delayed_covariance("OU", alpha, d, rho, t) + np.diag(op.sobs)
    Lc = np.linalg.cholesky(K)
    assert np.max(np.abs(f - z @ Lc.T)) < 1e-10 * np.max(np.abs(f))
    f2 = st.sample(seed=123, nsamples=3)
    assert np.array_equal(f, f2) and not np.array_equal(f, st.sample(seed=124, nsamples=3))
    zz = st.sample(seed=5, nsamples=500, return_z=True)[1].ravel()                 # 120 000 deviates
    assert abs(zz.mean()) < 0.01 and abs(zz.var() - 1.0) < 0.01 and abs(np.mean(zz ** 3)) < 0.03 and abs(np.mean(zz ** 4) - 3.0) < 0.06
    assert len(np.unique(zz)) == len(zz)
    big = st.sample(seed=9, nsamples=2000)
    emp = big.T @ big / 2000.0
    assert np.max(np.abs(emp - K)) < 0.25 * np.max(np.abs(K))                        # sample covariance -> K
    st.close()
    # simulator -> fit: the posterior over a small delay grid peaks at the simulated delay
    rg = np.random.default_rng(1)
    tt = [np.sort(rg.uniform(0, 60, 140)), np.sort(rg.uniform(0, 60, 120))]
    tt, yy, ss = gpcc_b200.simulatedata_device(tt, delays=[0.0, 3.0], alpha=[1.0, 1.5], b=[6.0, 15.0], rho=3.5, sigma=0.3, seed=4, ctx=ctx)
    assert [len(a) for a in yy] == [140, 120] and abs(np.mean(yy[1]) - 15.0) < 3.0
    cands = np.arange(0.0, 6.01, 0.5)
    res = gpcc_b200.gpccgrid(tt, yy, ss, np.stack([np.zeros_like(cands), cands], 1), kernel=gpcc_b200.OU, iterations=300, rhomax=50.0, ctx=ctx)
    assert abs(cands[np.argmax(res["posterior"])] - 3.0) <= 0.5


def test_random_problems_match_oracle(ctx):
    """Seeded sweep over random shapes: 1-5 bands of 2-90 points (total N from a handful to ~330, both paths, every residue of
    N modulo the 8-wide register tiles and the 128-wide HBM tiles that the sizes happen to hit), all four kernels, logL
    forward-only and with gradient against the oracle; plus one fitted candidate per problem against the oracle's L-BFGS."""
    rg = np.random.default_rng(2026)
    kernels = list(oracle.KERNELS)
    seen_paths = set()
    for trial in range(28):
        L = int(rg.integers(1, 6))
        nper = [int(v) for v in rg.integers(2, 91, L)]
        if trial % 7 == 0:
            nper = [int(v) for v in rg.integers(60, 120, 3)]                  # make sure the tiled path is visited
        L = len(nper)
        kernel = kernels[trial % 4]
        t, y, s, d = gpcc_b200.synthetic_bands(nper, seed=100 + trial, span=float(rg.uniform(8.0, 40.0)))
        op, p = oracle.Problem(t, y, s, kernel), Problem(t, y, s, kernel, ctx)
        M = 3
        delays = np.zeros((M, L)); delays[:, 1:] = rg.uniform(-4, 9, (M, L - 1))
        alpha, rho = rg.uniform(0.3, 3.0, (M, L)), np.exp(rg.uniform(np.log(0.3), np.log(60.0), M))
        ll, grad, info = p.loglik_batch(delays, alpha, rho, want_grad=True)
        seen_paths.add(ctx.stats()["path"])
        ll_f, info_f = p.loglik_batch(delays, alpha, rho)
        assert np.all(info == 0) and np.all(info_f == 0), (trial, nper, kernel)
        for m in range(M):
            rl, rgd = op.loglik_grad(delays[m], alpha[m], rho[m])
            assert abs(ll[m] - rl) <= LL_RTOL * abs(rl) and abs(ll_f[m] - rl) <= LL_RTOL * abs(rl), (trial, nper, kernel, m)
            assert np.max(np.abs(grad[m] - rgd)) <= GRAD_RTOL * max(np.max(np.abs(rgd)), 1e-3), (trial, nper, kernel, m)
        if trial % 4 == 0:
            th = gpcc_b200.initial_solutions(y, trial + 1, 1, 3, 0.1, 80.0)[0][0]
            r = p.fit_batch(delays[:1], th, iterations=400, rhomin=0.1, rhomax=80.0)
            o = oracle.gpcc(t, y, s, kernel=kernel, delays=delays[0], iterations=400, rhomin=0.1, rhomax=80.0, theta0=th[None], optimizer="lbfgs")
            # a scale that collapsed onto its 1e-8 floor (band decoupled from the latent process, SURVEY.md section 7) leaves logL
            # rising by ~1e-6 in total as theta_l -> -infinity: both optimisers sit in that degenerate valley and stop at
            # different depths; such candidates carry no posterior mass.  Everywhere else the 1e-6 contract is enforced.
            tol = 1e-5 if np.min(r["alpha"][0]) < 1e-6 else FIT_ATOL
            assert r["loglikel"][0] >= o[0] - tol, (trial, nper, kernel, r["loglikel"][0], o[0])
        p.close()
    assert seen_paths == {0, 1}


def test_path_crossover_sizes_match_oracle(ctx):
    """N = 199 is the largest problem of the fused register-resident path, N = 200 the smallest of the tiled path: both
    sides of the dispatch against the oracle (logL forward-only and with gradient), and a fit on each side."""
    for nper, path in (([70, 69, 60], 0), ([70, 70, 60], 1)):
        t, y, s, d = gpcc_b200.synthetic_bands(nper, seed=17)
        op, p = oracle.Problem(t, y, s, "matern52"), Problem(t, y, s, "matern52", ctx)
        rg = np.random.default_rng(6)
        delays = np.zeros((4, 3)); delays[:, 1:] = rg.uniform(0, 5, (4, 2))
        alpha, rho = rg.uniform(0.6, 2.5, (4, 3)), rg.uniform(1.0, 6.0, 4)
        ll, grad, info = p.loglik_batch(delays, alpha, rho, want_grad=True)
        assert ctx.stats()["path"] == path and np.all(info == 0)
        ll_f, _ = p.loglik_batch(delays, alpha, rho)
        for m in range(4):
            rl, rgd = op.loglik_grad(delays[m], alpha[m], rho[m])
            assert abs(ll[m] - rl) / abs(rl) < LL_RTOL and abs(ll_f[m] - rl) / abs(rl) < LL_RTOL
            assert np.max(np.abs(grad[m] - rgd)) / np.max(np.abs(rgd)) < GRAD_RTOL
        th = gpcc_b200.initial_solutions(y, 3, 1, 4, 0.1, 100.0)[0][0]
        r = p.fit_batch(delays[:2], th, iterations=300, rhomin=0.1, rhomax=100.0)
        for m in range(2):
            o = oracle.gpcc(t, y, s, kernel="matern52", delays=delays[m], iterations=300, rhomin=0.1, rhomax=100.0, theta0=th[None], optimizer="lbfgs")
            assert abs(r["loglikel"][m] - o[0]) < FIT_ATOL or r["loglikel"][m] > o[0]


def test_large_path_not_positive_definite_reports_leading_minor(ctx):
    t, y, s, d = gpcc_b200.synthetic_bands([200, 200], seed=2)
    t[1][150] = t[1][10]                                   # duplicated time stamp in band 2 (global index 350)
    s = [np.zeros(200), np.zeros(200)]                     # and no noise: exactly singular
    p = Problem(t, y, s, "rbf", ctx)
    ll, info = p.loglik_batch([[0.0, 0.0]], [[1.0, 1.0]], [0.05])
    assert ll[0] == -np.inf and 0 < info[0] <= 400


def test_large_path_fit_and_postb_pred(ctx):
    t, y, s, d = gpcc_b200.synthetic_bands([120, 110], seed=9)
    op, p = oracle.Problem(t, y, s, "matern32"), Problem(t, y, s, "matern32", ctx)
    theta0 = gpcc_b200.initial_solutions(y, 1, 1, 5, 0.1, 300.0)[0][0]
    delays = np.array([[0.0, 1.0], [0.0, 2.0], [0.0, 3.0]])
    res = p.fit_batch(delays, theta0, iterations=1000, rhomin=0.1, rhomax=300.0)
    for m in range(3):
        r = oracle.gpcc(t, y, s, kernel="matern32", delays=delays[m], iterations=1000, rhomax=300.0, theta0=theta0[None], optimizer="lbfgs")
        assert abs(res["loglikel"][m] - r[0]) < FIT_ATOL
    k = int(np.argmax(res["loglikel"]))
    mu, S = p.postb(delays[k], res["alpha"][k], res["rho"][k])
    omu, oS = op.postb(delays[k], res["alpha"][k], res["rho"][k])
    assert np.allclose(mu, omu, rtol=PRED_RTOL) and np.allclose(S, oS, rtol=PRED_RTOL)
    tt = np.linspace(0.0, 40.0, 33)
    m_, sd_, _, _ = p.predict(delays[k], res["alpha"][k], res["rho"][k], [tt, tt])
    om, osd = op.predict(delays[k], res["alpha"][k], res["rho"][k], tt)
    assert np.max(np.abs(m_ - np.concatenate(om)) / np.abs(np.concatenate(om))) < PRED_RTOL
    assert np.max(np.abs(sd_ - np.concatenate(osd)) / np.concatenate(osd)) < PRED_RTOL


@pytest.mark.parametrize("tag", ["n3072", "n6144"])
def test_cfg4_sizes_match_oracle_fixture(ctx, tag):
    """BASELINE config 4 (3 x 2048, matern52, N = 6144) and N = 3072 against the ORACLE: logL of the blocked Cholesky
    (forward) and of the symmetric sweep at 1e-10, gradient at 1e-8.  The oracle values (numpy potrf + potri, ~1 min at
    N = 6144) are committed in tests/golden/loglik_large.npz (tests/golden/make_golden_large.py); the data are regenerated
    from the seed and checked against the fixture's checksums."""
    g = load_golden("loglik_large")
    nper = [int(v) for v in g[tag + "_nper"]]
    t, y, s, d = gpcc_b200.synthetic_bands(nper, seed=int(g[tag + "_seed"]))
    assert np.allclose([a.sum() for a in t], g[tag + "_tsum"], rtol=1e-13) and np.allclose([a.sum() for a in y], g[tag + "_ysum"], rtol=1e-13)
    p = Problem(t, y, s, str(g["kernel"]), ctx)
    delays, alpha, rho = g[tag + "_delays"], g[tag + "_alpha"], g[tag + "_rho"]
    ll_f, info = p.loglik_batch(delays, alpha, rho)
    ll_s, grad, info2 = p.loglik_batch(delays, alpha, rho, want_grad=True)
    assert ctx.stats()["path"] == 1 and np.all(info == 0) and np.all(info2 == 0)
    assert np.max(np.abs(ll_f - g[tag + "_ll"]) / np.abs(g[tag + "_ll"])) < LL_RTOL
    assert np.max(np.abs(ll_s - g[tag + "_ll"]) / np.abs(g[tag + "_ll"])) < LL_RTOL
    assert np.max(np.abs(grad - g[tag + "_grad"]) / np.max(np.abs(g[tag + "_grad"]), axis=1, keepdims=True)) < GRAD_RTOL
    # the same candidate inside a fixed-theta sweep (3 tau_2 x 4 tau_3): shared leading block + last-band cache, same 1e-10
    sweep = np.array([[0.0, a, b] for a in (delays[0, 1], 2.4, 2.8) for b in (delays[0, 2], 4.6, 5.2, 5.8)])
    ll_w, info_w = p.loglik_batch(sweep, np.tile(alpha[0], (len(sweep), 1)), np.full(len(sweep), rho[0]))
    st = ctx.stats()
    assert np.all(info_w == 0) and st["n_tau_cache"] == len(sweep) and st["n_shared_prefix"] > 0
    assert abs(ll_w[0] - g[tag + "_ll"][0]) / abs(g[tag + "_ll"][0]) < LL_RTOL and abs(ll_w[0] - ll_f[0]) / abs(ll_f[0]) < 1e-14


def test_cfg4_size_properties(ctx):
    """Size-independent properties at N = 6144: permutation of points within a band leaves logL unchanged, and the analytic
    gradient agrees with a central finite difference of logL."""
    t, y, s, d = gpcc_b200.synthetic_bands([2048, 2048, 2048], seed=4)
    p = Problem(t, y, s, "matern52", ctx)
    delays = np.array([[0.0, 2.0, 4.0], [0.0, 7.4, 12.2]])
    alpha, rho = np.tile([1.0, 2.2, 4.0], (2, 1)), np.array([3.5, 2.0])
    ll_f, info = p.loglik_batch(delays, alpha, rho)
    ll_s, grad, info2 = p.loglik_batch(delays[:1], alpha[:1], rho[:1], want_grad=True)
    perm = [np.random.default_rng(l).permutation(2048) for l in range(3)]
    p2 = Problem([a[q] for a, q in zip(t, perm)], [a[q] for a, q in zip(y, perm)], s, "matern52", ctx)
    ll_p, _ = p2.loglik_batch(delays, alpha, rho)
    assert np.max(np.abs(ll_p - ll_f) / np.abs(ll_f)) < LL_RTOL
    rg = np.random.default_rng(0)
    v = rg.normal(size=4); v /= np.linalg.norm(v)
    h = 1e-4
    lp, _ = p.loglik_batch(delays[:1], alpha[:1] + h * v[:3], rho[:1] + h * v[3])
    lm, _ = p.loglik_batch(delays[:1], alpha[:1] - h * v[:3], rho[:1] - h * v[3])
    fd = (lp[0] - lm[0]) / (2 * h)
    assert abs(fd - grad[0] @ v) / abs(fd) < 1e-5


# ---- the fitted state behind postb / pred (gpcc_fit_state_*), against 50-digit arithmetic --------------------------------
@pytest.mark.parametrize("tag", ["a", "b"])
def test_pred_and_postb_match_exact_arithmetic(ctx, tag):
    """postb (:248-252) and predictTest (:259-307) against the 50-digit mpmath evaluation of the reference's formulas
    (tests/golden/pred_exact.npz, oracle/exact.py): means, standard deviations, the full predictive covariance and postb
    at north_star's 1e-8.  Case a = BASELINE config 1 (fused small-N fit path), case b = 230 points (tiled path)."""
    g = load_golden("pred_exact")
    idx = np.cumsum(g[tag + "_n"])[:-1]
    t, y, s = np.split(g[tag + "_t"], idx), np.split(g[tag + "_y"], idx), np.split(g[tag + "_s"], idx)
    tt = np.split(g[tag + "_ttest"], np.cumsum(g[tag + "_ntest"])[:-1])
    p = Problem(t, y, s, str(g[tag + "_kernel"]), ctx)
    st = p.fit_state(g[tag + "_delays"], g[tag + "_alpha"], float(g[tag + "_rho"]))
    mu_b, S_b = st.postb()
    assert np.max(np.abs(mu_b - g[tag + "_postb_mu"]) / np.abs(g[tag + "_postb_mu"])) < PRED_RTOL
    assert np.max(np.abs(S_b - g[tag + "_postb_Sigma"])) / np.max(np.abs(g[tag + "_postb_Sigma"])) < PRED_RTOL
    assert np.array_equal(S_b, S_b.T)
    mu, sd, S, nt = st.predict(tt, full_cov=True)
    assert np.max(np.abs(mu - g[tag + "_pred_mu"]) / np.abs(g[tag + "_pred_mu"])) < PRED_RTOL
    assert np.max(np.abs(sd - g[tag + "_pred_sd"]) / g[tag + "_pred_sd"]) < PRED_RTOL
    assert np.max(np.abs(S - g[tag + "_pred_Sigma"])) / np.max(np.abs(g[tag + "_pred_Sigma"])) < PRED_RTOL
    assert np.array_equal(S, S.T)
    # the stateless entry points go through the same cached factor and return the same bits
    mu2, sd2, _, _ = p.predict(g[tag + "_delays"], g[tag + "_alpha"], float(g[tag + "_rho"]), tt)
    mu_b2, S_b2 = p.postb(g[tag + "_delays"], g[tag + "_alpha"], float(g[tag + "_rho"]))
    assert np.array_equal(mu2, mu) and np.array_equal(sd2, sd) and np.array_equal(mu_b2, mu_b) and np.array_equal(S_b2, S_b)


def test_fit_state_factorises_once_and_handles_many_test_points(ctx):
    """The closure state (:235-252) is built once: any number of pred calls, of any size, reuse the factor (the reference
    re-factorises KSobsB on every call, :275, :283).  70 000 test points exceed a CUDA grid's y-dimension."""
    t, y, s, d = gpcc_b200.synthetic_bands([12, 9], seed=21, span=10.0)
    op, p = oracle.Problem(t, y, s, "OU"), Problem(t, y, s, "OU", ctx)
    alpha, rho = np.array([1.3, 0.8]), 2.0
    st = p.fit_state(d, alpha, rho)
    om, osd = op.predict(d, alpha, rho, np.linspace(0.0, 10.0, 7))
    for _ in range(3):
        m_, sd_, _, _ = st.predict([np.linspace(0.0, 10.0, 7)] * 2)
        assert np.allclose(m_, np.concatenate(om), rtol=PRED_RTOL) and np.allclose(sd_, np.concatenate(osd), rtol=PRED_RTOL)
    big = np.linspace(-5.0, 15.0, 35000)
    mb, sdb, _, _ = st.predict([big, big])
    assert mb.shape == (70000,) and np.all(np.isfinite(mb)) and np.all(sdb > 0)
    pick = np.array([0, 1234, 34999])
    om, osd = op.predict(d, alpha, rho, big[pick])
    assert np.allclose(mb[pick], om[0], rtol=PRED_RTOL) and np.allclose(mb[35000 + pick], om[1], rtol=PRED_RTOL)
    assert np.allclose(sdb[pick], osd[0], rtol=PRED_RTOL) and np.allclose(sdb[35000 + pick], osd[1], rtol=PRED_RTOL)
    ll, info = st.predict_loglik([[1.0, 2.0], [3.0]], [[6.0, 6.5], [15.0]], [[0.3, 0.3], [0.4]])
    ref = op.predict_loglik(d, alpha, rho, [[1.0, 2.0], [3.0]], [[6.0, 6.5], [15.0]], [[0.3, 0.3], [0.4]])
    assert info == 0 and abs(ll - ref) / abs(ref) < PRED_RTOL
    assert st.factorisations == 1
    with pytest.raises(gpcc_b200.GpccError):
        p.fit_state(d, [1.0, -1.0], rho)                     # all(scale .> 0) (delayedCovariance.jl:3)
    st.close()
    ctx2 = gpcc_b200.Context(1)                              # destroy order: context first, then state and problem (finalizers)
    p2 = Problem(t, y, s, "OU", ctx2)
    st2 = p2.fit_state(d, alpha, rho)
    ctx2.close(); st2.close(); p2.close()


# ---- edge cases of the batched entry points ---------------------------------------------------------------------
def test_single_band_and_eight_bands(ctx):
    # L = 1 is the reference's `singlegp` (src/util.jl:74-78); L = 8 is GPCC_MAX_BANDS
    for nper, kernel in (([25], "matern32"), ([9, 8, 7, 6, 9, 8, 7, 6], "OU")):
        t, y, s, d = gpcc_b200.synthetic_bands(nper, seed=11, span=15.0)
        L = len(nper)
        op, p = oracle.Problem(t, y, s, kernel), Problem(t, y, s, kernel, ctx)
        rg = np.random.default_rng(4)
        delays = np.zeros((5, L)); delays[:, 1:] = rg.uniform(-3, 6, (5, L - 1))
        alpha, rho = rg.uniform(0.5, 2.0, (5, L)), rg.uniform(0.5, 6.0, 5)
        ll, grad, info = p.loglik_batch(delays, alpha, rho, want_grad=True)
        for m in range(5):
            rl, rgd = op.loglik_grad(delays[m], alpha[m], rho[m])
            assert abs(ll[m] - rl) / abs(rl) < LL_RTOL and np.max(np.abs(grad[m] - rgd)) / np.max(np.abs(rgd)) < GRAD_RTOL
        th = gpcc_b200.initial_solutions(y, 2, 1, 3, 0.1, 50.0)[0][0]
        r = p.fit_batch(delays[:2], th, iterations=200, rhomin=0.1, rhomax=50.0)
        for m in range(2):
            o = oracle.gpcc(t, y, s, kernel=kernel, delays=delays[m], iterations=200, rhomin=0.1, rhomax=50.0, theta0=th[None], optimizer="lbfgs")
            assert r["loglikel"][m] >= o[0] - FIT_ATOL      # same optimum or a better basin
    with pytest.raises(gpcc_b200.GpccError):
        Problem([np.arange(3.0)] * 9, [np.arange(3.0)] * 9, [np.ones(3)] * 9, "OU", ctx)     # more than GPCC_MAX_BANDS


def test_large_batches_are_chunked_consistently(ctx):
    """More evaluations than one staging chunk (2^18): results must not depend on where the chunk boundaries fall."""
    t, y, s, d = gpcc_b200.synthetic_bands([7, 2, 13], seed=6, span=10.0)
    p = Problem(t, y, s, "OU", ctx)
    M = (1 << 18) + 1234
    rg = np.random.default_rng(8)
    delays = np.zeros((M, 3)); delays[:, 1:] = rg.uniform(0, 5, (M, 2))
    alpha, rho = rg.uniform(0.3, 3.0, (M, 3)), rg.uniform(0.2, 50.0, M)
    ll, info = p.loglik_batch(delays, alpha, rho)
    pick = np.r_[0:50, (1 << 18) - 25:(1 << 18) + 25, M - 50:M]
    ll_s, _ = p.loglik_batch(delays[pick], alpha[pick], rho[pick])
    assert np.array_equal(ll[pick], ll_s) and np.all(info == 0)
    op = oracle.Problem(t, y, s, "OU")
    for m in (0, 1 << 18, M - 1):
        assert abs(ll[m] - op.loglik(delays[m], alpha[m], rho[m])) / abs(ll[m]) < LL_RTOL
    # a fitted grid with 60 000 candidates: screening runs in several chunks (2^18 / P candidates each)
    th = gpcc_b200.initial_solutions(y, 1, 1, 5, 0.1, 100.0)[0][0]
    Mf = 60000
    r = p.grid_posterior(delays[:Mf], th, iterations=50, rhomin=0.1, rhomax=100.0)
    r2 = p.fit_batch(delays[Mf - 100:Mf], th, iterations=50, rhomin=0.1, rhomax=100.0)
    assert np.array_equal(r["loglikel"][Mf - 100:], r2["loglikel"]) and abs(r["posterior"].sum() - 1.0) < 1e-10


def test_prior_with_minus_infinity_and_iteration_cap_zero(ctx):
    g = load_golden("fit_cfg1_cfg2")
    p = Problem(g["tb"], g["yb"], g["sb"], "matern32", ctx)
    delays = np.stack([np.zeros(11), np.linspace(0, 10, 11)], 1)
    lp = np.zeros(11); lp[[0, 5]] = -np.inf
    r = p.grid_posterior(delays, g["theta0"], iterations=1000, rhomin=0.1, rhomax=300.0, logprior=lp)
    assert r["posterior"][0] == 0.0 and r["posterior"][5] == 0.0 and abs(r["posterior"].sum() - 1.0) < 1e-12
    r0 = p.fit_batch(delays[:3], g["theta0"], iterations=0, rhomin=0.1, rhomax=300.0)     # screening only (:207-209)
    scr = np.max(np.stack([p.loglik_theta_batch(delays[:3], np.tile(th, (3, 1)), 0.1, 300.0)[0] for th in g["theta0"]]), axis=0)
    assert np.allclose(r0["loglikel"], scr, rtol=1e-14) and np.all(r0["info"] == 1) and np.all(r0["nfev"] == 5)


@pytest.mark.parametrize("switch", [
    {"GPCC_FIT_HOST": "1"},                                    # host-driven batched L-BFGS (api.cu fit_shard) instead of the persistent fit kernel
    {"GPCC_SMALL_VARIANT": "0"},                               # one CTA per SM at 255 registers whatever the batch size
], ids=lambda d: "+".join(f"{k[5:]}={v}" for k, v in d.items()))
def test_alternative_drivers_agree(ctx, switch):
    """The A/B switches of the fused small-N path (read once per process) must give the same answers as the default path:
    golden log-likelihoods and gradients, LAPACK-style info on a singular matrix, the fitted cfg1 optimum and the cfg2
    posterior against the golden fixture."""
    import os, subprocess, sys
    code = (
        "import numpy as np, sys; sys.path.insert(0, %r)\n"
        "import gpcc_b200, oracle\n"
        "from conftest import load_golden\n"
        "for name in ('loglik_3band_matern32', 'loglik_2band_OU', 'loglik_ragged_OU', 'loglik_3x64_matern52'):\n"
        "    g = load_golden(name)\n"
        "    p = gpcc_b200.Problem(g['tb'], g['yb'], g['sb'], g['kernel'])\n"
        "    ll, grad, info = p.loglik_batch(g['delays'], g['alpha'], g['rho'], want_grad=True)\n"
        "    assert np.all(info == 0)\n"
        "    assert np.max(np.abs(ll - g['loglik']) / np.abs(g['loglik'])) < 1e-10, name\n"
        "    assert np.max(np.abs(grad - g['grad']) / np.max(np.abs(g['grad']), axis=1, keepdims=True)) < 1e-8, name\n"
        "    ll2, info2 = p.loglik_batch(g['delays'][:3], g['alpha'][:3], g['rho'][:3])\n"
        "    assert np.array_equal(ll2, ll[:3]), name\n"
        "t = [np.array([1.0, 1.0, 2.0, 3.0]), np.array([1.5, 2.5, 2.5])]; y = [np.array([1.0, 2.0, 1.5, 0.5]), np.array([3.0, 2.0, 2.5])]\n"
        "p = gpcc_b200.Problem(t, y, [np.zeros(4), np.zeros(3)], 'rbf')      # duplicated times, zero noise: singular\n"
        "ll, grad, info = p.loglik_batch([[0.0, 0.0]], [[1.0, 1.0]], [1.0], want_grad=True)\n"
        "assert info[0] > 0 and ll[0] == -np.inf and np.all(grad == 0.0), (ll, info)\n"
        "ll, info = p.loglik_batch([[0.0, 0.0]], [[1.0, 1.0]], [1.0])\n"
        "assert info[0] > 0 and ll[0] == -np.inf, (ll, info)\n"
        "g = load_golden('fit_cfg1_cfg2')\n"
        "loglikel, pred, (alpha, postb, rho) = gpcc_b200.gpcc(g['tb'], g['yb'], g['sb'], kernel=gpcc_b200.matern32, delays=g['truedelays'],\n"
        "                                                    iterations=1000, rhomax=300, theta0=g['theta0'], verbose=False)\n"
        "assert abs(loglikel - float(g['loglikel'])) < 1e-6\n"
        "p = gpcc_b200.Problem(g['tb'], g['yb'], g['sb'], 'matern32')\n"
        "delays = np.stack([np.zeros_like(g['cands']), g['cands']], 1)\n"
        "res = p.grid_posterior(delays, g['theta0'], iterations=1000, rhomin=0.1, rhomax=300.0)\n"
        "assert np.max(np.abs(res['loglikel'] - g['ll_grid'])[g['post_flat'] > 1e-12]) < 1e-6\n"
        "assert np.max(np.abs(res['posterior'] - g['post_flat'])) < 1e-4\n"
        "r0 = p.fit_batch(delays[:3], g['theta0'], iterations=0, rhomin=0.1, rhomax=300.0)\n"
        "assert np.all(r0['info'] == 1) and np.all(r0['nfev'] == 5)\n"
        "print('VARIANT-OK')\n"
    ) % os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, PYTHONPATH=os.path.dirname(os.path.abspath(__file__)), **switch)
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "VARIANT-OK" in r.stdout, (r.stdout[-500:], r.stderr[-2500:])


def test_device_resident_fit_equals_host_driven_loop(ctx):
    """The persistent fit kernel (small_fit.cu) and the host-driven batched L-BFGS (api.cu) run the same state machine
    (lbfgs.h) on the same evaluator: optima agree far inside the 1e-6 contract (not bitwise: the transforms use the device's
    exp/log1p/tanh in one and glibc's in the other), evaluation counts agree up to the odd line-search trial."""
    import os, subprocess, sys, json
    code = (
        "import numpy as np, sys, json; sys.path.insert(0, %r)\n"
        "import gpcc_b200\n"
        "t, y, s, d = gpcc_b200.simulatethreelightcurves()\n"
        "p = gpcc_b200.Problem(t, y, s, 'matern32')\n"
        "c = np.arange(0.0, 20.0001, 1.0)\n"
        "delays = np.array([[0.0, a, b] for b in c for a in c])\n"
        "th = gpcc_b200.initial_solutions(y, 1, 1, 5, 0.1, 300.0)[0][0]\n"
        "r = p.fit_batch(delays, th, iterations=1000, rhomin=0.1, rhomax=300.0)\n"
        "print('RESULT' + json.dumps(dict(ll=r['loglikel'].tolist(), nfev=r['nfev'].tolist(), info=r['info'].tolist())))\n"
    ) % os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = {}
    for tag, extra in (("device", {}), ("host", {"GPCC_FIT_HOST": "1"})):
        r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, **extra), capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        out[tag] = json.loads([l for l in r.stdout.splitlines() if l.startswith("RESULT")][0][6:])
    lld, llh = np.array(out["device"]["ll"]), np.array(out["host"]["ll"])
    nd, nh = np.array(out["device"]["nfev"]), np.array(out["host"]["nfev"])
    gap = np.abs(lld - llh)
    print("device vs host loop: max gap %.2e, candidates beyond 1e-6: %d of %d; mean nfev %.1f vs %.1f, identical counts %.0f %%"
          % (gap.max(), np.sum(gap > 1e-6), len(gap), nd.mean(), nh.mean(), 100 * np.mean(nd == nh)))
    assert np.median(gap) < 1e-9 and np.sum(gap > 1e-6) <= len(gap) // 50      # a different basin is possible where the surface is flat
    assert abs(nd.mean() - nh.mean()) < 0.05 * nh.mean()
