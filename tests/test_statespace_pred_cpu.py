"""The fit state of the state-space method without a GPU: the reference route of tests/ss_pred_reference.py (an RTS smoother
over training and test points, and the test log-likelihood as a difference of two Kalman filters) against the dense oracle
and against the 50-digit fixture, and the per-point formula of gpcc_b200/csrc/ss_model.h (ss::point_moments, built with g++)
against an RTS step with explicit inverses."""
import os
import shutil
import subprocess

import numpy as np
import pytest

import oracle
from oracle import statespace as ss
from conftest import load_golden, ROOT
from ss_pred_reference import make_test_times, predict_loglik, smooth_predict

FIXTURES = ["loglik_2band_OU", "loglik_2band_matern32", "loglik_2band_matern52", "loglik_3band_OU",
            "loglik_3band_matern32", "loglik_3band_matern52", "loglik_ragged_OU", "loglik_3x64_matern52"]


@pytest.mark.parametrize("name", FIXTURES)
def test_smoother_matches_dense_oracle(name):
    g = load_golden(name)
    pr = oracle.Problem(g["tb"], g["yb"], g["sb"], g["kernel"])
    rng = np.random.default_rng(FIXTURES.index(name))
    for j in range(min(3, len(g["rho"]))):
        d, a, r = g["delays"][j], g["alpha"][j], float(g["rho"][j])
        tt = make_test_times(g["tb"], rng)
        mu, sd = smooth_predict(pr, g["kernel"], d, a, r, tt)
        rm, rS = pr.predict_full(d, a, r, tt)
        rsd = np.sqrt(np.maximum(np.diag(rS), 1e-6))
        assert np.max(np.abs(mu - rm)) <= 1e-9 * np.max(np.abs(rm)), (name, j)
        assert np.max(np.abs(sd - rsd) / rsd) <= 1e-9, (name, j)
        yt = [pr.mub[l] + rng.standard_normal(len(x)) for l, x in enumerate(tt)]
        st = [0.1 + 0.2 * rng.random(len(x)) for x in tt]
        ll = predict_loglik(pr, g["kernel"], d, a, r, tt, yt, st)
        rl = pr.predict_loglik(d, a, r, tt, yt, st)
        assert abs(ll - rl) <= 1e-9 * abs(rl), (name, j, ll, rl)


@pytest.mark.parametrize("tag", ["a", "b"])
def test_smoother_against_exact_fixture(tag):
    g = load_golden("pred_exact")
    idx = np.cumsum(g[tag + "_n"])[:-1]
    t, y, s = np.split(g[tag + "_t"], idx), np.split(g[tag + "_y"], idx), np.split(g[tag + "_s"], idx)
    tt = np.split(g[tag + "_ttest"], np.cumsum(g[tag + "_ntest"])[:-1])
    kernel = str(g[tag + "_kernel"])
    mu, sd = smooth_predict(oracle.Problem(t, y, s, kernel), kernel, g[tag + "_delays"], g[tag + "_alpha"],
                            float(g[tag + "_rho"]), tt)
    assert np.max(np.abs(mu - g[tag + "_pred_mu"]) / np.abs(g[tag + "_pred_mu"])) < 1e-8
    assert np.max(np.abs(sd - g[tag + "_pred_sd"]) / g[tag + "_pred_sd"]) < 1e-8


# ---- ss::point_moments (host build of ss_model.h) ---------------------------------------------------------------------
@pytest.fixture(scope="module")
def point_exe(tmp_path_factory):
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    exe = str(tmp_path_factory.mktemp("ss_point") / "ss_point_host_test")
    subprocess.run(["g++", "-O2", "-std=c++17", "-I", os.path.join(ROOT, "gpcc_b200", "csrc"),
                    os.path.join(ROOT, "tests", "host", "ss_point_host_test.cpp"), "-o", exe], check=True)
    return exe


def _spd(rng, n, scale):
    X = rng.standard_normal((n, n))
    return scale * (X @ X.T / n + 0.1 * np.eye(n))


def _packed(M):
    return np.concatenate([M[i, i:] for i in range(M.shape[0])])


@pytest.mark.parametrize("kernel", ["OU", "matern32", "matern52"])
def test_point_moments_against_rts_step(point_exe, kernel):
    """Random filtered moments at step i and smoothed moments at step i+1: the adjoint form of ss::point_moments against the
    RTS step m* = m_f + G (m_s - m-), P* = P_f + G (P_s - P-) G', G = P_f A2' inv(P-), with m_f, P_f predicted over dt1."""
    rng = np.random.default_rng(3)
    kid = {"OU": 0, "matern32": 2, "matern52": 3}[kernel]
    lines, refs = [], []
    for L in (1, 3, 8):
        for rho, dt1, dt2, later in ((2.0, 0.3, 0.7, 1), (0.5, 0.0, 0.2, 1), (40.0, 1.5, 0.01, 1), (3.0, 0.4, 0.0, 0)):
            d = ss.sde(kernel, rho)[0].shape[0]
            D = d + L
            l, a = int(rng.integers(L)), 0.5 + rng.random()
            m, P = rng.standard_normal(D), _spd(rng, D, 1.0)
            P[d:, d:] += np.diag(rng.uniform(0.5, 50.0, L))
            T1, T2 = np.eye(D), np.eye(D)
            Q1, Q2 = np.zeros((D, D)), np.zeros((D, D))
            if dt1 > 0:
                A, Q, _, _ = ss.transition(kernel, rho, dt1)
                T1[:d, :d], Q1[:d, :d] = A, Q
            mf, Pf = T1 @ m, T1 @ P @ T1.T + Q1
            h = np.zeros(D)
            h[0], h[d + l] = a, 1.0
            line = "%d %d %d %.17g %.17g %.17g %d %.17g\n" % (kid, L, l, a, rho, dt1, later, dt2)
            line += " ".join("%.17g" % v for v in np.concatenate([m, _packed(P)]))
            if later:
                A, Q, _, _ = ss.transition(kernel, rho, dt2)
                T2[:d, :d], Q2[:d, :d] = A, Q
                mm, Pm = T2 @ mf, T2 @ Pf @ T2.T + Q2
                Ps = Pm - 0.5 * Pm @ _spd(rng, D, 0.3) @ Pm / np.linalg.norm(Pm) ** 2 * np.linalg.norm(Pm)
                Ps = 0.5 * (Ps + Ps.T)
                ms = mm + 0.3 * rng.standard_normal(D)
                Pi = np.linalg.inv(Pm)
                lam, Lam = Pi @ (mm - ms), Pi @ (Pm - Ps) @ Pi
                line += " " + " ".join("%.17g" % v for v in np.concatenate([lam, _packed(0.5 * (Lam + Lam.T))]))
                G = Pf @ T2.T @ Pi
                mstar, Pstar = mf + G @ (ms - mm), Pf + G @ (Ps - Pm) @ G.T
            else:
                mstar, Pstar = mf, Pf
            lines.append(line + "\n")
            refs.append((h @ mstar, h @ Pstar @ h, (kernel, L, rho, dt1, dt2, later)))
    out = subprocess.run([point_exe], input="".join(lines), check=True, capture_output=True, text=True).stdout.split("\n")
    for line, (rm, rv, where) in zip(out, refs):
        mean, var = (float(x) for x in line.split())
        assert abs(mean - rm) <= 1e-10 * max(1.0, abs(rm)), (where, mean, rm)
        assert abs(var - rv) <= 1e-10 * abs(rv), (where, var, rv)
    assert len([x for x in out if x.strip()]) == len(refs)
