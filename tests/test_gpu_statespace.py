"""The state-space method (Problem(..., method="statespace"), gpcc_problem_set_method) on the device: the Kalman filter
against the golden fixtures, against the dense method on the same data, and against oracle/statespace.py beyond the reach
of a dense factorisation; info, fits, postb, the lazy fit state behind `pred`, and determinism."""
import numpy as np
import pytest

import gpcc_b200
import oracle
from gpcc_b200 import Problem
from oracle import statespace as ss
from conftest import load_golden

pytestmark = pytest.mark.gpu

LL_RTOL = 1e-10
GRAD_RTOL = 1e-8
FIXTURES = ["loglik_2band_OU", "loglik_2band_matern32", "loglik_2band_matern52", "loglik_3band_OU",
            "loglik_3band_matern32", "loglik_3band_matern52", "loglik_ragged_OU", "loglik_3x64_matern52"]


def _check(ll, grad, rl, rg, where):
    for m in range(len(rl)):
        assert abs(ll[m] - rl[m]) <= LL_RTOL * abs(rl[m]), (where, m, ll[m], rl[m])
        if grad is not None:
            assert np.max(np.abs(grad[m] - rg[m])) <= GRAD_RTOL * np.max(np.abs(rg[m])), (where, m, grad[m], rg[m])


@pytest.mark.parametrize("name", FIXTURES)
def test_golden_fixtures(ctx, name):
    g = load_golden(name)
    p = Problem(g["tb"], g["yb"], g["sb"], g["kernel"], ctx, method="statespace")
    ll, grad, info = p.loglik_batch(g["delays"], g["alpha"], g["rho"], want_grad=True)
    assert np.all(info == 0)
    _check(ll, grad, g["loglik"], g["grad"], name)
    assert ctx.stats()["path"] == 2
    ll0, info0 = p.loglik_batch(g["delays"], g["alpha"], g["rho"])
    assert np.all(info0 == 0)
    _check(ll0, None, g["loglik"], None, name)


@pytest.mark.parametrize("N", [3072, 6144])
def test_golden_large(ctx, N):
    g = load_golden("loglik_large")
    k = "n%d_" % N
    t, y, s, _ = gpcc_b200.synthetic_bands([int(v) for v in g[k + "nper"]], seed=int(g[k + "seed"]))
    assert np.allclose([a.sum() for a in t], g[k + "tsum"]) and np.allclose([a.sum() for a in y], g[k + "ysum"])
    p = Problem(t, y, s, str(g["kernel"]), ctx, method="statespace")
    ll, grad, info = p.loglik_batch(g[k + "delays"], g[k + "alpha"], g[k + "rho"], want_grad=True)
    assert np.all(info == 0)
    _check(ll, grad, g[k + "ll"], g[k + "grad"], N)


def _edge_data(rng):
    """Unsorted times, duplicates inside a band, shifted times that coincide across bands (with the delays below)."""
    t0 = np.sort(rng.uniform(0, 40, 60))
    t = [rng.permutation(np.concatenate([t0, t0[::7]])), t0[:50] + 3.0, np.sort(rng.uniform(0, 40, 45))]
    y = [np.sin(a / 4.0) + 0.3 * rng.standard_normal(len(a)) for a in t]
    s = [0.2 + 0.1 * rng.random(len(a)) for a in t]
    return t, y, s


def _batch(rng, M, L, coincident):
    delays = np.zeros((M, L))
    delays[:, 1:] = rng.uniform(-5, 20, (M, L - 1))
    delays[: M // 4, 1] = coincident                        # shifted band 1 lands exactly on band 0
    alpha = rng.uniform(0.5, 2.5, (M, L))
    rho = np.exp(rng.uniform(np.log(0.1), np.log(300.0), M))
    rho[:2] = [0.1, 300.0][:M]
    return delays, alpha, rho


@pytest.mark.parametrize("kernel", ["OU", "matern32", "matern52"])
def test_agrees_with_dense_method(ctx, kernel):
    rng = np.random.default_rng(7)
    t, y, s = _edge_data(rng)
    pd = Problem(t, y, s, kernel, ctx)
    ps = Problem(t, y, s, kernel, ctx, method="statespace")
    for M in (1, 31, 148, 149, 1000):
        delays, alpha, rho = _batch(rng, M, 3, 3.0)
        for want_grad in (False, True):
            rd = pd.loglik_batch(delays, alpha, rho, want_grad=want_grad)
            rs = ps.loglik_batch(delays, alpha, rho, want_grad=want_grad)
            assert np.all(rd[-1] == 0) and np.all(rs[-1] == 0)
            _check(rs[0], rs[1] if want_grad else None, rd[0], rd[1] if want_grad else None, (kernel, M, want_grad))
    # switching back gives the dense path's bits
    pd2 = Problem(t, y, s, kernel, ctx, method="statespace")
    pd2.set_method("dense")
    a = pd.loglik_batch(delays[:5], alpha[:5], rho[:5], want_grad=True)
    b = pd2.loglik_batch(delays[:5], alpha[:5], rho[:5], want_grad=True)
    assert all(np.array_equal(u, v) for u, v in zip(a, b))


@pytest.mark.parametrize("L", [1, 8])
def test_band_counts_against_dense(ctx, L):
    rng = np.random.default_rng(11 + L)
    t = [np.sort(rng.uniform(0, 30, 2 if l == L - 1 and L > 1 else 20)) for l in range(L)]   # one band of 2 points
    y = [np.cos(a / 3.0) + 0.3 * rng.standard_normal(len(a)) for a in t]
    s = [0.25 * np.ones(len(a)) for a in t]
    delays, alpha, rho = _batch(rng, 40, L, 0.0) if L > 1 else (np.zeros((40, 1)), rng.uniform(0.5, 2, (40, 1)),
                                                                  np.exp(rng.uniform(np.log(0.1), np.log(300.0), 40)))
    for kernel in ("OU", "matern32", "matern52"):
        rd = Problem(t, y, s, kernel, ctx).loglik_batch(delays, alpha, rho, want_grad=True)
        rs = Problem(t, y, s, kernel, ctx, method="statespace").loglik_batch(delays, alpha, rho, want_grad=True)
        _check(rs[0], rs[1], rd[0], rd[1], (kernel, L))


@pytest.mark.parametrize("kernel", ["OU", "matern32"])
def test_beyond_dense_reach(ctx, kernel):
    """N = 3 x 32768: a dense factorisation would need 77 GB; the filter against the numpy filter of the oracle."""
    t, y, s, d = gpcc_b200.synthetic_bands([32768] * 3, seed=3, span=4000.0)
    p = Problem(t, y, s, kernel, ctx, method="statespace")
    op = oracle.Problem(t, y, s, kernel)
    delays = np.array([d, d + [0.0, 1.5, -2.0], d + [0.0, -3.0, 4.5]])
    alpha = np.array([[1.0, 1.3, 0.8], [0.7, 1.1, 1.6], [1.4, 0.9, 1.2]])
    rho = np.array([2.0, 15.0, 120.0])
    ll, grad, info = p.loglik_batch(delays, alpha, rho, want_grad=True)
    assert np.all(info == 0)
    ref = [ss.filter(op, kernel, delays[m], alpha[m], rho[m], want_grad=True) for m in range(3)]
    _check(ll, grad, [r[0] for r in ref], [r[1] for r in ref], kernel)


def test_info_and_errors(ctx):
    # zero noise on a duplicated time: after the first point, the second is known exactly and its innovation variance is
    # 0.  The band's values make Sigma_b exactly 3 and alpha = 1, so every step of the update is exact: S = 0 at step 2.
    t, y, s = [np.array([1.0, 1.0])], [np.array([0.0, 0.2449489742783178])], [np.zeros(2)]
    p = Problem(t, y, s, "OU", ctx, method="statespace")
    assert p.Sigmab[0] == 3.0
    ll, grad, info = p.loglik_batch([[0.0]], [[1.0]], [1.0], want_grad=True)
    assert info[0] == 2 and ll[0] == -np.inf and np.all(grad == 0.0)
    g = load_golden("loglik_3band_OU")
    p = Problem(g["tb"], g["yb"], g["sb"], "OU", ctx, method="statespace")
    ll, info = p.loglik_batch([[0.0, 1.0, 2.0]] * 3, [[1.0, -1.0, 1.0], [1.0, 1.0, 1.0], [np.nan, 1.0, 1.0]], [1.0, 0.0, 1.0])
    assert np.all(info == -1) and np.all(ll == -np.inf)
    with pytest.raises(gpcc_b200.GpccError):
        Problem(g["tb"], g["yb"], g["sb"], "rbf", ctx, method="statespace")
    with pytest.raises(gpcc_b200.GpccError):
        p.set_method("kalman")
    theta0 = gpcc_b200.initial_solutions(g["yb"], 1, 1, 5, 0.1, 20.0)[0][0]
    with pytest.raises(gpcc_b200.GpccError):
        p.fit_batch(g["delays"][:2], theta0, iterations=10, rhomin=0.1, rhomax=20.0, optimizer="neldermead")


def test_grid_fit_against_golden(ctx):
    g = load_golden("fit_cfg1_cfg2")
    tb, yb, sb = g["tb"], g["yb"], g["sb"]
    delays = np.stack([np.zeros_like(g["cands"]), g["cands"]], 1)
    res = gpcc_b200.gpccgrid(tb, yb, sb, delays, kernel=gpcc_b200.matern32, iterations=1000, rhomax=300.0,
                             theta0=g["theta0"], ctx=ctx, method="statespace")
    assert ctx.stats()["path"] == 2
    mass = g["post_flat"] > 1e-12
    assert np.max(np.abs(res["loglikel"][mass] - g["ll_grid"][mass])) < 1e-6
    assert np.max(np.abs(res["posterior"] - g["post_flat"])) < 1e-4


def test_postb_and_lazy_fit_state(ctx):
    g = load_golden("loglik_3band_matern52")
    p = Problem(g["tb"], g["yb"], g["sb"], g["kernel"], ctx, method="statespace")
    for j in range(4):
        mu, S = p.postb(g["delays"][j], g["alpha"][j], g["rho"][j])
        fmu, fS = p.fit_state(g["delays"][j], g["alpha"][j], g["rho"][j]).postb()
        assert np.max(np.abs(mu - fmu)) <= 1e-10 * np.max(np.abs(fmu)) and np.max(np.abs(S - fS)) <= 1e-10 * np.max(np.abs(fS))
    t, y, s, d = gpcc_b200.synthetic_bands([8192] * 3, seed=4, span=1500.0)
    theta0 = gpcc_b200.initial_solutions(y, 1, 1, 3, 0.1, 20.0)[0]
    ll, pred, (alpha, postb, rho) = gpcc_b200.gpcc(t, y, s, kernel=gpcc_b200.matern32, delays=d, iterations=20,
                                                   rhomax=20.0, theta0=theta0, ctx=ctx, verbose=False,
                                                   method="statespace")
    assert ctx.stats()["path"] == 2
    assert np.isfinite(ll) and np.all(np.isfinite(alpha)) and np.isfinite(rho)
    assert np.all(np.isfinite(postb.mean)) and np.all(np.isfinite(postb.cov))
    assert pred._state is None                                    # no dense factorisation so far
    # a small problem to exercise the lazy state through pred
    g = load_golden("fit_cfg1_cfg2")
    ll, pred, (alpha, postb, rho) = gpcc_b200.gpcc(g["tb"], g["yb"], g["sb"], kernel=gpcc_b200.matern32,
                                                   delays=g["truedelays"], iterations=1000, rhomax=300.0,
                                                   theta0=g["theta0"], ctx=ctx, verbose=False, method="statespace")
    assert pred._state is None
    mu_, sd_ = pred(g["ttest"])
    assert pred._state is not None and pred.state.factorisations == 1
    fmu, fS = pred.state.postb()
    assert np.allclose(postb.mean, fmu, rtol=1e-10) and np.allclose(postb.cov, fS, rtol=1e-10)
    assert abs(ll - float(g["loglikel"])) < 1e-6
    assert np.allclose(np.concatenate(mu_), g["pred_mu"].ravel(), rtol=1e-5, atol=1e-6)


def test_bitwise_deterministic(ctx):
    rng = np.random.default_rng(5)
    t, y, s = _edge_data(rng)
    p = Problem(t, y, s, "matern52", ctx, method="statespace")
    delays, alpha, rho = _batch(rng, 300, 3, 3.0)
    a = p.loglik_batch(delays, alpha, rho, want_grad=True)
    b = p.loglik_batch(delays, alpha, rho, want_grad=True)
    assert all(np.array_equal(u, v) for u, v in zip(a, b))


def test_two_devices_bitwise_equal_one():
    import gpcc_b200._lib  # noqa: F401
    try:
        import torch
        n = torch.cuda.device_count()
    except Exception:
        n = 1
    if n < 2:
        pytest.skip("needs two GPUs")
    g = load_golden("fit_cfg1_cfg2")
    delays = np.stack([np.zeros_like(g["cands"]), g["cands"]], 1)
    out = []
    for nd in (1, 2):
        c = gpcc_b200.Context(nd)
        p = Problem(g["tb"], g["yb"], g["sb"], "matern32", c, method="statespace")
        out.append(p.grid_posterior(delays, g["theta0"], iterations=1000, rhomin=0.1, rhomax=300.0))
    for k in ("loglikel", "posterior", "theta", "nfev", "info"):
        assert np.array_equal(out[0][k], out[1][k]), k
