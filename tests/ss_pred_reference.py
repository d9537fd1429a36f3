"""Reference route for the fit state of the state-space method (gpcc_ss_state_*, StateSpaceFitState): a numpy RTS smoother
over the training points merged with the test points, and the test log-likelihood as the difference of two runs of the
Kalman filter of oracle/statespace.py.  Built on that module's expm transitions (a different route from the device's closed
forms and its Bryson-Frazier backward pass); test infrastructure only."""
import numpy as np

from oracle.model import JITTER, SIGMA_FLOOR
from oracle.statespace import filter, sde, transition


# ---- predictions of a fitted state (the device's state-space fit state, gpcc_ss_state_*) ------------------------------
class Data:
    """What the filter and the smoother read of an oracle.Problem (mu_b = mean, Sigma_b = 100 var), without its N x N
    matrices: for N beyond a dense reference."""

    def __init__(self, tarray, yarray, stdarray):
        self.t = [np.asarray(a, dtype=np.float64) for a in tarray]
        self.y = [np.asarray(a, dtype=np.float64) for a in yarray]
        self.s = [np.asarray(a, dtype=np.float64) for a in stdarray]
        self.L = len(self.t)
        self.n = np.array([len(a) for a in self.t])
        self.N = int(self.n.sum())
        self.band = np.repeat(np.arange(self.L), self.n)
        self.Y, self.sobs = np.concatenate(self.y), np.concatenate(self.s) ** 2
        self.mub = np.array([a.mean() for a in self.y])
        self.Sigmab = 100.0 * np.array([a.var(ddof=1) for a in self.y])


def _prior(kernel, rho, problem):
    _, _, Pinf, _ = sde(kernel, rho)
    d = Pinf.shape[0]
    P = np.zeros((d + problem.L, d + problem.L))
    P[:d, :d] = Pinf
    P[d:, d:] = np.diag(problem.Sigmab)
    return P, d


def smooth_predict(problem, kernel, delays, alpha, rho, ttest):
    """Per-point predictive means and standard deviations (sqrt(max(var + JITTER, SIGMA_FLOOR)), as pred(ttest) of the dense
    route): an RTS smoother over the training points merged with the test points (ttest: one array per band), the test
    points as predict-only steps that sit after training points at the same shifted time.  Explicit inverses, expm
    transitions.  Returns (mu, sd) in the input order of the concatenated test points."""
    pr = problem
    L = pr.L
    P0, d = _prior(kernel, rho, pr)
    D = d + L
    tt = [np.asarray(a, dtype=np.float64) for a in ttest]
    steps = []                                          # (shifted time, is test, band, index)
    s_tr = [pr.t[l] - delays[l] for l in range(L)]
    r = pr.Y - pr.mub[pr.band]
    off = np.concatenate([[0], np.cumsum(pr.n)])
    for l in range(L):
        steps += [(s_tr[l][i], 0, l, off[l] + i) for i in range(len(s_tr[l]))]
    k = 0
    for l in range(L):
        for i in range(len(tt[l])):
            steps.append((tt[l][i] - delays[l], 1, l, k))
            k += 1
    steps.sort(key=lambda x: (x[0], x[1], x[2], x[3]))
    n = len(steps)
    m, P = np.zeros(D), P0.copy()
    mp, Pp, mf, Pf, Tm = [], [], [], [], []
    prev = None
    for s, is_test, l, i in steps:
        T = np.eye(D)
        if prev is not None and s != prev:
            A, Q, _, _ = transition(kernel, rho, s - prev)
            T[:d, :d] = A
            m = T @ m
            P = T @ P @ T.T
            P[:d, :d] += Q
        prev = s
        mp.append(m.copy()); Pp.append(P.copy()); Tm.append(T)
        if not is_test:
            h = np.zeros(D)
            h[0], h[d + l] = alpha[l], 1.0
            Ph = P @ h
            S = h @ Ph + pr.sobs[i]
            m = m + Ph * (r[i] - h @ m) / S
            P = P - np.outer(Ph, Ph) / S
            P = 0.5 * (P + P.T)
        mf.append(m.copy()); Pf.append(P.copy())
    ms, Ps = mf[-1], Pf[-1]
    out_m, out_v = np.empty(k), np.empty(k)
    for j in range(n - 1, -1, -1):
        if j < n - 1:
            G = Pf[j] @ Tm[j + 1].T @ np.linalg.inv(Pp[j + 1])
            ms = mf[j] + G @ (ms - mp[j + 1])
            Ps = Pf[j] + G @ (Ps - Pp[j + 1]) @ G.T
            Ps = 0.5 * (Ps + Ps.T)
        s, is_test, l, i = steps[j]
        if is_test:
            h = np.zeros(D)
            h[0], h[d + l] = alpha[l], 1.0
            out_m[i] = pr.mub[l] + h @ ms
            out_v[i] = h @ Ps @ h
    return out_m, np.sqrt(np.maximum(out_v + JITTER, SIGMA_FLOOR))


class _Merged:
    """Training points followed, per band, by test points (noise sigmatest^2 + JITTER), under the training prior of b."""

    def __init__(self, pr, ttest, ytest, stest):
        self.L = pr.L
        self.t = [np.concatenate([pr.t[l], np.asarray(ttest[l], dtype=np.float64)]) for l in range(pr.L)]
        y = [np.concatenate([pr.y[l], np.asarray(ytest[l], dtype=np.float64)]) for l in range(pr.L)]
        s2 = [np.concatenate([pr.s[l] ** 2, np.asarray(stest[l], dtype=np.float64) ** 2 + JITTER]) for l in range(pr.L)]
        self.n = np.array([len(a) for a in self.t])
        self.N = int(self.n.sum())
        self.band = np.repeat(np.arange(pr.L), self.n)
        self.Y, self.sobs = np.concatenate(y), np.concatenate(s2)
        self.mub, self.Sigmab = pr.mub, pr.Sigmab


def predict_loglik(problem, kernel, delays, alpha, rho, ttest, ytest, stest):
    """Test log-likelihood logpdf(N(mu_pred, Sigma_pred + diag(sigmatest^2)), ytest) (Sigma_pred with the JITTER) as the
    difference of two filters: training and test points together, minus the training points alone."""
    ll_all = filter(_Merged(problem, ttest, ytest, stest), kernel, delays, alpha, rho)[0]
    return ll_all - filter(problem, kernel, delays, alpha, rho)[0]


def make_test_times(t, rng, n_between=6):
    """Per band: before the first and after the last training time, exactly on training times (one of them twice), and
    n_between unsorted points in between."""
    out = []
    for tl in t:
        lo, hi = tl.min(), tl.max()
        pts = [lo - 3.0, hi + 2.5, tl[len(tl) // 2], tl[len(tl) // 2], tl[0]] + list(rng.uniform(lo, hi, n_between))
        out.append(rng.permutation(np.array(pts)))
    return out
