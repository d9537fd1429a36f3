"""A numpy route to the posterior draws of the state-space fit state (gpcc_ss_state_sample, StateSpaceFitState.sample), test
infrastructure beside the tests.  The draw is affine in its deviates z (per sample: d+1 per merged point, training points in
input order then test points in input order, then L shift deviates): draw = offset + M z.  The prior part comes from
tests/ss_sample_reference.sample_map over the training and test times merged (training first on ties, test points with
sigma^2 = 1e-8), the shifts add sqrt(Sigma_b) z_b, and the conditioning is a dense solve with K + Sobs + B, so that
offset = mu_pred and M M' = Sigma_pred of oracle.model.Problem.predict_full when the route is right."""
from types import SimpleNamespace

import numpy as np

from oracle.covariance import delayed_covariance
from oracle.model import JITTER
from ss_sample_reference import DIM, sample_map


def post_map(pr, kernel, delays, alpha, rho, ttest):
    """(offset [NT], M [NT][(N+NT)(d+1) + L]) of the draw for the oracle.Problem pr and test times ttest (one array per band)."""
    L, N, d = pr.L, pr.N, DIM[kernel]
    S = d + 1
    tt = [np.asarray(a, dtype=np.float64) for a in ttest]
    nt = np.array([len(a) for a in tt])
    NT = int(nt.sum())
    NM = N + NT
    # merged problem, band-major (training of band l, then its test points), and the device index of each of its points
    off_tr = np.concatenate([[0], np.cumsum(pr.n)])
    off_te = np.concatenate([[0], np.cumsum(nt)])
    t = [np.concatenate([pr.t[l], tt[l]]) for l in range(L)]
    dev = np.concatenate([np.concatenate([off_tr[l] + np.arange(pr.n[l]), N + off_te[l] + np.arange(nt[l])]) for l in range(L)])
    n = np.array([len(a) for a in t])
    sobs = np.concatenate([np.concatenate([pr.s[l] ** 2, np.full(nt[l], JITTER)]) for l in range(L)])
    mp = SimpleNamespace(t=t, L=L, N=NM, n=n, band=np.repeat(np.arange(L), n), sobs=sobs)
    Mm = sample_map(mp, kernel, delays, alpha, rho)               # [NM][NM S], band-major on both sides
    Mf = np.zeros((NM, NM * S))                                   # the same map, device order on both sides
    cols = (dev[:, None] * S + np.arange(S)[None, :]).ravel()
    Mf[np.ix_(dev, cols)] = Mm
    K = NM * S + L
    bt = np.repeat(np.arange(L), nt)
    Zb = np.zeros((L, K))
    Zb[:, NM * S:] = np.diag(np.sqrt(pr.Sigmab))                  # b~' as a function of z
    Y = np.hstack([Mf[:N], np.zeros((N, L))]) + Zb[pr.band]       # prior draw of the data, y~'
    G = np.hstack([Mf[N:], np.zeros((NT, L))]) + Zb[bt]           # prior draw at the test points minus mu_b
    KSB = pr.Ktilde(delays, alpha, rho)
    Bs = np.where(pr.band[:, None] == bt[None, :], pr.Sigmab[pr.band][:, None], 0.0)
    kBs = delayed_covariance(kernel, alpha, delays, rho, pr.t, tt) + Bs
    H = np.linalg.solve(KSB, kBs).T                               # Cov(g*, y) Cov(y)^-1
    r = pr.Y - pr.bbar
    return pr.mub[bt] + H @ r, G - H @ Y


def make_test_times(rng, t, empty_band):
    """Per band: times before, after and between the band's training times, and equal to three of them; no test point in
    band empty_band.  Unsorted."""
    out = []
    for l, a in enumerate(t):
        if l == empty_band:
            out.append(np.empty(0))
            continue
        u = np.concatenate([[a.min() - 7.0, a.min() - 0.5, a.max() + 0.3, a.max() + 9.0],
                            rng.uniform(a.min(), a.max(), 5), a[rng.integers(len(a), size=3)]])
        out.append(rng.permutation(u))
    return out
