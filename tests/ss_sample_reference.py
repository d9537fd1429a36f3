"""A numpy route to the O(N) draw of gpcc_ss_sample (test infrastructure, beside the tests so that the oracle package stays
as it is).  Transition and process noise come from oracle.statespace (scipy expm, Q = P_inf - A P_inf A'), the merged order
from oracle.statespace.merge_order, the stationary factor from numpy's Cholesky and each step's from `factor`.  sample_map
returns the linear map M from the deviates [N][d+1] (input order: d process deviates, then one noise deviate per point) to
the draw f, so that M M' is the covariance of the draw."""
import numpy as np

from oracle import statespace as oss

DIM = {"OU": 1, "matern32": 2, "matern52": 3}


def factor(Q):
    """C with C C' = Q.  Q = P_inf - A P_inf A' is accurate to eps |P_inf| only, and at small lambda D its tiny entries are
    noise that may make it slightly indefinite, so that neither a plain nor a scaled Cholesky factor is reliable there: a
    symmetric eigen-factor with negative eigenvalues clamped to zero keeps C C' - Q at the size of that noise.  M M' does not
    depend on which factor is used; the lower Cholesky factor of gpcc_ss_sample is checked where Q is accurate."""
    w, V = np.linalg.eigh(0.5 * (Q + Q.T))
    return V * np.sqrt(np.maximum(w, 0.0))


def sample_map(problem, kernel, delays, alpha, rho):
    """M [N][N (d+1)]: f = M z for the deviates z [N][d+1] flattened, f and z in the problem's input order."""
    order, s = oss.merge_order(problem, delays)
    _, _, Pinf, _ = oss.sde(kernel, rho)
    d = DIM[kernel]
    S = d + 1
    N = problem.N
    sig = np.sqrt(problem.sobs)
    M = np.zeros((N, N * S))
    X = np.zeros((d, N * S))                 # the f-state as a linear function of the deviates
    prev = None
    for k, i in enumerate(order):
        cols = slice(i * S, i * S + d)
        if k == 0:
            X[:, cols] = np.linalg.cholesky(Pinf)
        elif s[i] != prev:                   # a tie adds no process noise
            A, Q, _, _ = oss.transition(kernel, rho, s[i] - prev)
            X = A @ X
            X[:, cols] += factor(Q)
        prev = s[i]
        M[i] = alpha[problem.band[i]] * X[0]
        M[i, i * S + d] += sig[i]
    return M


def data(rng, L):
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
