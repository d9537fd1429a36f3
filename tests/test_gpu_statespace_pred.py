"""The fit state of the state-space method (Problem.statespace_fit_state, gpcc_ss_state_*) on the device: per-point means and
standard deviations and the test log-likelihood against the 50-digit fixture, against the dense fit state on the same data,
and against the reference route of tests/ss_pred_reference.py beyond the reach of a dense factorisation; large calls,
reproducibility, errors, lifetime, ABI and a K-fold score."""
import ctypes as C

import numpy as np
import pytest

import gpcc_b200
import oracle
from gpcc_b200 import Problem, _lib
from conftest import load_golden
from ss_pred_reference import Data, make_test_times, smooth_predict

pytestmark = pytest.mark.gpu

RTOL = 1e-8


def _split(g, tag):
    idx = np.cumsum(g[tag + "_n"])[:-1]
    return np.split(g[tag + "_t"], idx), np.split(g[tag + "_y"], idx), np.split(g[tag + "_s"], idx)


@pytest.mark.parametrize("tag", ["a", "b"])
def test_exact_fixture(ctx, tag):
    g = load_golden("pred_exact")
    t, y, s = _split(g, tag)
    tt = np.split(g[tag + "_ttest"], np.cumsum(g[tag + "_ntest"])[:-1])
    p = Problem(t, y, s, str(g[tag + "_kernel"]), ctx, method="statespace")
    st = p.statespace_fit_state(g[tag + "_delays"], g[tag + "_alpha"], float(g[tag + "_rho"]))
    mu, sd, S, nt = st.predict(tt)
    assert S is None and list(nt) == list(g[tag + "_ntest"])
    assert np.max(np.abs(mu - g[tag + "_pred_mu"]) / np.abs(g[tag + "_pred_mu"])) < RTOL
    assert np.max(np.abs(sd - g[tag + "_pred_sd"]) / g[tag + "_pred_sd"]) < RTOL


def _data(rng, L):
    """Unsorted bands with duplicated times; band 1 is band 0 shifted by 3 (coincident shifted times at delay 3)."""
    t0 = np.sort(rng.uniform(0, 40, 40))
    t = [rng.permutation(np.concatenate([t0, t0[::6]]))]
    if L > 1:
        t.append(rng.permutation(t0[:30] + 3.0))
    for _ in range(2, L):
        t.append(np.sort(rng.uniform(-5, 45, 25)))
    y = [np.sin(a / 4.0) + 0.3 * rng.standard_normal(len(a)) + 2.0 * l for l, a in enumerate(t)]
    s = [0.2 + 0.1 * rng.random(len(a)) for a in t]
    delays = np.concatenate([[0.0], [3.0] if L > 1 else [], np.linspace(-2.0, 6.0, max(L - 2, 0))])
    return t, y, s, delays


@pytest.mark.parametrize("kernel", ["OU", "matern32", "matern52"])
@pytest.mark.parametrize("L", [1, 2, 3, 8])
@pytest.mark.parametrize("rho", [0.1, 300.0])
def test_agrees_with_dense_fit_state(ctx, kernel, L, rho):
    rng = np.random.default_rng(100 * L + int(rho))
    t, y, s, delays = _data(rng, L)
    alpha = 0.6 + rng.random(L)
    pd = Problem(t, y, s, kernel, ctx)
    ps = Problem(t, y, s, kernel, ctx, method="statespace")
    fd = pd.fit_state(delays, alpha, rho)
    fs = ps.statespace_fit_state(delays, alpha, rho)
    tt = make_test_times(t, rng)
    if L > 1:
        tt[1] = np.empty(0)                                     # a band without test points
    mu, sd, _, _ = fs.predict(tt)
    rm, rsd, _, _ = fd.predict(tt)
    where = (kernel, L, rho)
    assert np.max(np.abs(mu - rm)) <= RTOL * np.max(np.abs(rm)), where
    assert np.max(np.abs(sd - rsd) / rsd) <= RTOL, where
    yt = [m + 0.3 * rng.standard_normal(len(m)) for m in np.split(rm, np.cumsum([len(a) for a in tt])[:-1])]
    stt = [0.1 + 0.2 * rng.random(len(a)) for a in tt]
    ll, info = fs.predict_loglik(tt, yt, stt)
    rl, rinfo = fd.predict_loglik(tt, yt, stt)
    assert info == 0 and rinfo == 0
    assert abs(ll - rl) <= RTOL * abs(rl), (where, ll, rl)
    empty = [np.empty(0)] * L
    mu0, sd0, _, nt0 = fs.predict(empty)
    assert mu0.shape == (0,) and sd0.shape == (0,) and nt0.sum() == 0
    assert fs.predict_loglik(empty, empty, empty) == (0.0, 0)


def test_beyond_dense_reach(ctx):
    """N = 3 x 32768: a dense fit state would need 77 GB; against the RTS smoother of the reference route."""
    t, y, s, d = gpcc_b200.synthetic_bands([32768] * 3, seed=3, span=4000.0)
    p = Problem(t, y, s, "matern32", ctx, method="statespace")
    alpha, rho = np.array([1.0, 1.3, 0.8]), 15.0
    st = p.statespace_fit_state(d, alpha, rho)
    rng = np.random.default_rng(9)
    tt = [np.concatenate([rng.uniform(a.min() - 20, a.max() + 20, 100), a[rng.integers(len(a), size=5)]]) for a in t]
    mu, sd, _, _ = st.predict(tt)
    rm, rsd = smooth_predict(Data(t, y, s), "matern32", d, alpha, rho, tt)
    assert np.max(np.abs(mu - rm)) <= RTOL * np.max(np.abs(rm))
    assert np.max(np.abs(sd - rsd) / rsd) <= RTOL


def test_large_call_equals_split_calls_and_states_reproduce(ctx):
    t, y, s, d = gpcc_b200.synthetic_bands([3000, 2500, 2000], seed=5, span=300.0)
    p = Problem(t, y, s, "matern52", ctx, method="statespace")
    alpha, rho = np.array([1.2, 0.9, 1.6]), 7.0
    st = p.statespace_fit_state(d, alpha, rho)
    rng = np.random.default_rng(2)
    big = [rng.uniform(-20, 320, n) for n in (30000, 25000, 15000)]
    mu, sd, _, _ = st.predict(big)
    assert mu.shape == (70000,)
    parts = [st.predict([b[k // 3::4] if l == k % 3 else np.empty(0) for l, b in enumerate(big)]) for k in range(12)]
    mu2, sd2 = np.empty_like(mu), np.empty_like(sd)
    off = np.concatenate([[0], np.cumsum([len(b) for b in big])])
    for k, (m_, s_, _, _) in enumerate(parts):
        l = k % 3
        idx = off[l] + np.arange(len(big[l]))[k // 3::4]
        mu2[idx], sd2[idx] = m_, s_
    assert np.array_equal(mu, mu2) and np.array_equal(sd, sd2)
    st2 = p.statespace_fit_state(d, alpha, rho)
    mu3, sd3, _, _ = st2.predict(big)
    assert np.array_equal(mu, mu3) and np.array_equal(sd, sd3)
    yt = [rng.standard_normal(200) for _ in range(3)]
    sg = [0.3 * np.ones(200) for _ in range(3)]
    tt = [b[:200] for b in big]
    assert st.predict_loglik(tt, yt, sg) == st2.predict_loglik(tt, yt, sg)


def test_errors(ctx):
    g = load_golden("loglik_3band_matern32")
    d, a, r = g["delays"][0], g["alpha"][0], float(g["rho"][0])
    dense = Problem(g["tb"], g["yb"], g["sb"], g["kernel"], ctx)
    with pytest.raises(gpcc_b200.GpccError):
        dense.statespace_fit_state(d, a, r)
    p = Problem(g["tb"], g["yb"], g["sb"], g["kernel"], ctx, method="statespace")
    for aa, rr in ((np.array([1.0, -1.0, 1.0]), r), (np.array([1.0, np.nan, 1.0]), r), (a, 0.0), (a, np.inf)):
        with pytest.raises(gpcc_b200.GpccError):
            p.statespace_fit_state(d, aa, rr)
    st = p.statespace_fit_state(d, a, r)
    tt = [np.array([1.0, 2.0]), np.array([np.nan]), np.array([3.0])]
    with pytest.raises(gpcc_b200.GpccError):
        st.predict(tt)
    ok = [np.array([1.0, 2.0]), np.array([1.5]), np.array([3.0])]
    with pytest.raises(gpcc_b200.GpccError):
        st.predict_loglik(ok, [np.zeros(2), np.zeros(1), np.zeros(1)], [np.ones(2), -np.ones(1), np.ones(1)])
    with pytest.raises(gpcc_b200.GpccError):
        st.predict(ok, full_cov=True)
    with pytest.raises(gpcc_b200.GpccError):
        st.pred(ok)                                             # Vector{Vector}: (mu, Sigma) needs the dense state
    mu_, sd_ = st.pred(np.array([1.0, 2.0, 3.0]))               # Vector: per band (mu, sigma)
    assert len(mu_) == 3 and all(len(m) == 3 for m in mu_) and all(np.all(x > 0) for x in sd_)
    assert st.pred(ok, [np.zeros(2), np.zeros(1), np.zeros(1)], [np.ones(2), np.ones(1), np.ones(1)]) == \
        st.predict_loglik(ok, [np.zeros(2), np.zeros(1), np.zeros(1)], [np.ones(2), np.ones(1), np.ones(1)])[0]
    lib = _lib.load()
    h = C.c_void_p()
    nt = np.array([-1, 0, 0], dtype=np.int32)
    assert lib.gpcc_ss_state_predict(st._h, nt.ctypes.data_as(C.POINTER(C.c_int)), None, None, None) < 0
    # zero noise on a duplicated time: the second innovation variance is exactly 0 (as in test_gpu_statespace)
    z = Problem([np.array([1.0, 1.0])], [np.array([0.0, 0.2449489742783178])], [np.zeros(2)], "OU", ctx, method="statespace")
    dd, aa = np.zeros(1), np.ones(1)
    rc = lib.gpcc_ss_state_create(z._h, dd.ctypes.data_as(C.POINTER(C.c_double)), aa.ctypes.data_as(C.POINTER(C.c_double)),
                                  1.0, C.byref(h))
    assert rc == -6 and not h.value


def test_outlives_its_problem(ctx):
    g = load_golden("loglik_3band_OU")
    p = Problem(g["tb"], g["yb"], g["sb"], "OU", ctx, method="statespace")
    st = p.statespace_fit_state(g["delays"][1], g["alpha"][1], float(g["rho"][1]))
    tt = make_test_times(g["tb"], np.random.default_rng(4))
    yt = [np.ones(len(a)) for a in tt]
    sg = [0.5 * np.ones(len(a)) for a in tt]
    before = st.predict(tt)[:2], st.predict_loglik(tt, yt, sg)
    p.set_method("dense")
    p.close()
    after = st.predict(tt)[:2], st.predict_loglik(tt, yt, sg)
    assert all(np.array_equal(u, v) for u, v in zip(before[0], after[0])) and before[1] == after[1]


def test_abi():
    lib = _lib.load()
    assert lib.gpcc_version() == 103
    for name in ("gpcc_ss_state_create", "gpcc_ss_state_destroy", "gpcc_ss_state_predict", "gpcc_ss_state_predict_loglik"):
        assert hasattr(lib, name) and name in _lib.EXPORTS


def test_kfold_score_at_fixed_theta(ctx):
    """performcv's fold score (the test log-likelihood of the held-out part) at fixed hyper-parameters: the state-space
    fit state per fold against the dense fit state."""
    g = load_golden("fit_cfg1_cfg2")
    t, y, s = g["tb"], g["yb"], g["sb"]
    folds = gpcc_b200.cv_folds([len(a) for a in t], 5, 1)
    delays, alpha, rho = g["truedelays"], np.array([1.0, 2.0]), 2.0
    for k in range(5):
        tr = [f != k for f in folds]
        part = lambda arrs, masks: [np.asarray(a)[m] for a, m in zip(arrs, masks)]
        te = [~m for m in tr]
        ps = Problem(part(t, tr), part(y, tr), part(s, tr), "matern32", ctx, method="statespace")
        pd = Problem(part(t, tr), part(y, tr), part(s, tr), "matern32", ctx)
        ll, info = ps.statespace_fit_state(delays, alpha, rho).predict_loglik(part(t, te), part(y, te), part(s, te))
        rl, rinfo = pd.fit_state(delays, alpha, rho).predict_loglik(part(t, te), part(y, te), part(s, te))
        assert info == 0 and rinfo == 0 and abs(ll - rl) <= RTOL * abs(rl), (k, ll, rl)
