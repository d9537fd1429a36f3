"""Joint posterior draws of the state-space fit state (StateSpaceFitState.sample, gpcc_ss_state_sample) on the device: the
exact map from deviates to draws against the dense predictive distribution, the mean against the state's own predictions up
to N ~ 1e5, the moments of generator draws at N ~ 3e5, reproducibility, edge cases, argument checks and lifetime."""
import ctypes as C

import numpy as np
import pytest

import gpcc_b200
from gpcc_b200 import Problem, _lib
from oracle.model import Problem as OracleProblem
from ss_post_sample_reference import make_test_times
from ss_sample_reference import DIM, data

pytestmark = pytest.mark.gpu

_dp, _ip = C.POINTER(C.c_double), C.POINTER(C.c_int)


def _ndev(N, NT, kernel, L):
    return (N + NT) * (DIM[kernel] + 1) + L


@pytest.mark.parametrize("kernel", ["OU", "matern32", "matern52"])
@pytest.mark.parametrize("L", [1, 2, 3, 8])
@pytest.mark.parametrize("rho", [0.1, 300.0])
def test_exact_map(ctx, kernel, L, rho):
    """z = the identity: the draws minus the z = 0 draw are the columns of the map M, M M' = Sigma_pred and the z = 0 draw is
    mu_pred of the dense oracle.  Test times before, after, between and on training times, one band without test points."""
    rng = np.random.default_rng(10 * L + int(rho))
    t, y, s, delays = data(rng, L)
    alpha = 0.6 + rng.random(L)
    tt = make_test_times(rng, t, 1 if L > 1 else -1)
    p = Problem(t, y, s, kernel, ctx, method="statespace")
    st = p.statespace_fit_state(delays, alpha, rho)
    NT = sum(len(a) for a in tt)
    K = _ndev(p.N, NT, kernel, L)
    g0 = st.sample(tt, 0, nsamples=1, z=np.zeros((1, K)))[0]
    G = st.sample(tt, 0, nsamples=K, z=np.eye(K))
    M = (G - g0).T
    mu, S = OracleProblem(t, y, s, kernel).predict_full(delays, alpha, rho, tt)
    err = np.max(np.abs(M @ M.T - S)) / np.max(np.diag(S))
    assert err <= 1e-9, (kernel, L, rho, err)
    assert np.max(np.abs(g0 - mu)) <= 1e-9 * np.max(np.abs(mu)), (kernel, L, rho)


@pytest.mark.parametrize("n", [[2500] * 3, [32768] * 3])
def test_zero_deviates_give_the_predictive_mean(ctx, n):
    """z = 0: the draw is the smoother mean of the residuals, equal to the state's own predict mean (up to N = 3 x 32768,
    beyond a dense reference)."""
    t, y, s, d = gpcc_b200.synthetic_bands(n, seed=3, span=n[0] / 8.0)
    p = Problem(t, y, s, "matern32", ctx, method="statespace")
    alpha, rho = np.array([1.0, 1.3, 0.8]), 15.0
    st = p.statespace_fit_state(d, alpha, rho)
    rng = np.random.default_rng(9)
    tt = [np.concatenate([rng.uniform(a.min() - 20, a.max() + 20, 100), a[rng.integers(len(a), size=5)]]) for a in t]
    NT = sum(len(a) for a in tt)
    g = st.sample(tt, 0, z=np.zeros((1, _ndev(p.N, NT, "matern32", 3))))[0]
    mu = st.predict(tt)[0]
    assert np.max(np.abs(g - mu)) <= 1e-10 * np.max(np.abs(mu))


def test_moments_at_scale(ctx):
    """N = 3 x 100 000, 4 000 generator draws at 51 test times: sample mean within 5 sd / sqrt(n) of predict, sample variance
    within 5 of its standard errors of sd^2."""
    t, y, s, d = gpcc_b200.synthetic_bands([100000] * 3, seed=7, span=20000.0)
    p = Problem(t, y, s, "matern32", ctx, method="statespace")
    alpha, rho = np.array([1.0, 1.3, 0.8]), 15.0
    st = p.statespace_fit_state(d, alpha, rho)
    rng = np.random.default_rng(1)
    tt = [np.concatenate([rng.uniform(-50.0, 20050.0, 15), [-200.0, 20300.0]]) for _ in range(3)]
    n = 4000
    g = st.sample(tt, 11, nsamples=n)
    mu, sd, _, _ = st.predict(tt)
    assert g.shape == (n, 51)
    assert np.all(np.abs(g.mean(0) - mu) <= 5.0 * sd / np.sqrt(n))
    assert np.all(np.abs(g.var(0, ddof=1) - sd ** 2) <= 5.0 * sd ** 2 * np.sqrt(2.0 / (n - 1)))


def test_reproducible(ctx):
    rng = np.random.default_rng(5)
    t, y, s, delays = data(rng, 3)
    p = Problem(t, y, s, "matern52", ctx, method="statespace")
    st = p.statespace_fit_state(delays, np.array([1.0, 0.7, 1.4]), 3.0)
    tt = make_test_times(rng, t, -1)
    a = st.sample(tt, 42, nsamples=7)
    assert np.array_equal(a, st.sample(tt, 42, nsamples=7))
    assert np.array_equal(a[:1], st.sample(tt, 42, nsamples=1))
    f, z = st.sample(tt, 42, nsamples=7, return_z=True)
    assert np.array_equal(f, a) and z.shape == (7, _ndev(p.N, a.shape[1], "matern52", 3))
    assert np.array_equal(st.sample(tt, 0, nsamples=7, z=z), a)
    b = st.sample(tt, 43, nsamples=7)
    assert not np.any(a == b)
    st2 = p.statespace_fit_state(delays, np.array([1.0, 0.7, 1.4]), 3.0)
    assert np.array_equal(st2.sample(tt, 42, nsamples=7), a)


def test_edge_cases(ctx):
    """NT = 0 writes nothing; the draws follow the order of the test times (unsorted, on training times)."""
    rng = np.random.default_rng(6)
    t, y, s, delays = data(rng, 2)
    p = Problem(t, y, s, "OU", ctx, method="statespace")
    st = p.statespace_fit_state(delays, np.array([1.0, 0.7]), 2.0)
    g = st.sample([np.empty(0), np.empty(0)], 1, nsamples=3)
    assert g.shape == (3, 0)
    tt = [t[0][[5, 1, 5, 9]], np.array([30.0, -3.0, t[1][2]])]
    a = st.sample(tt, 1, nsamples=4)
    perm0, perm1 = np.array([3, 0, 2, 1]), np.array([1, 2, 0])
    K = _ndev(p.N, 7, "OU", 2)
    z = np.random.default_rng(0).standard_normal((4, K))
    g = st.sample(tt, 0, nsamples=4, z=z)
    # the same draws with the test points given in another order: permute their deviates alongside
    S, N = 2, p.N
    zt = z[:, N * S:7 * S + N * S].reshape(4, 7, S)
    order = np.concatenate([perm0, 4 + perm1])
    z2 = np.concatenate([z[:, :N * S], zt[:, order].reshape(4, 7 * S), z[:, -2:]], axis=1)
    tt2 = [tt[0][perm0], tt[1][perm1]]
    g2 = st.sample(tt2, 0, nsamples=4, z=z2)
    assert np.max(np.abs(g2 - g[:, order])) <= 1e-12 * np.max(np.abs(g))
    assert g[:, 0].std() > 0 and np.all(np.isfinite(a))


def test_errors(ctx):
    rng = np.random.default_rng(8)
    t, y, s, delays = data(rng, 2)
    p = Problem(t, y, s, "matern32", ctx, method="statespace")
    st = p.statespace_fit_state(delays, np.array([1.0, 0.7]), 2.0)
    lib = _lib.load()
    nt = np.array([2, 1], dtype=np.int32)
    tt = np.array([1.0, 2.0, 3.0])
    f = np.empty((2, 3))
    K = _ndev(p.N, 3, "matern32", 2)

    def call(h=st._h, n=nt, x=tt, ns=2, z=None, out=f):
        return lib.gpcc_ss_state_sample(h, None if n is None else n.ctypes.data_as(_ip),
                                        None if x is None else x.ctypes.data_as(_dp), 1, ns,
                                        None if z is None else z.ctypes.data_as(_dp), None if out is None else out.ctypes.data_as(_dp),
                                        None)

    assert call() == 0
    assert call(h=None) == -1 and call(n=None) == -1 and call(x=None) == -1 and call(out=None) == -1
    assert call(x=np.array([1.0, np.inf, 3.0])) == -3
    assert call(n=np.array([-1, 1], dtype=np.int32)) == -5
    assert call(ns=0) == -7
    assert call(n=np.array([1 << 30, 1], dtype=np.int32), x=None) == -7
    z = np.zeros(2 * K)
    assert call(z=z) == 0
    z[K + 3] = np.nan
    assert call(z=z) == -8
    with pytest.raises(gpcc_b200.GpccError):
        st.sample([np.array([1.0]), np.array([2.0])], 0, z=np.zeros((1, K)))        # wrong z shape


def test_outlives_its_problem(ctx):
    rng = np.random.default_rng(4)
    t, y, s, delays = data(rng, 3)
    p = Problem(t, y, s, "matern52", ctx, method="statespace")
    st = p.statespace_fit_state(delays, np.array([1.0, 0.7, 1.4]), 3.0)
    tt = make_test_times(rng, t, 2)
    before = st.sample(tt, 3, nsamples=5)
    p.set_method("dense")
    p.close()
    assert np.array_equal(st.sample(tt, 3, nsamples=5), before)
