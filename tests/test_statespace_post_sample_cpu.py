"""The posterior draws of the state-space fit state without a GPU: the affine map of tests/ss_post_sample_reference.py from the
deviates to the draws has offset mu_pred and M M' = Sigma_pred of the dense oracle, and ss::point_mean_weights of
gpcc_b200/csrc/ss_model.h (built with g++) gives the smoothed mean of ss::point_moments as a linear function of m and lam."""
import os
import shutil
import subprocess

import numpy as np
import pytest

import oracle
from conftest import ROOT
from ss_post_sample_reference import make_test_times, post_map
from ss_sample_reference import DIM, data


@pytest.mark.parametrize("kernel", ["OU", "matern32", "matern52"])
@pytest.mark.parametrize("L", [1, 2, 3, 8])
@pytest.mark.parametrize("rho", [0.1, 300.0])
def test_map_moments_are_predictive_moments(kernel, L, rho):
    rng = np.random.default_rng(10 * L + int(rho))
    t, y, s, delays = data(rng, L)
    alpha = 0.6 + rng.random(L)
    pr = oracle.Problem(t, y, s, kernel)
    tt = make_test_times(rng, t, 1 if L > 1 else -1)
    off, M = post_map(pr, kernel, delays, alpha, rho, tt)
    mu, S = pr.predict_full(delays, alpha, rho, tt)
    NT = len(mu)
    assert M.shape == (NT, (pr.N + NT) * (DIM[kernel] + 1) + L)
    scale = np.max(np.diag(S))
    assert np.max(np.abs(M @ M.T - S)) <= 1e-10 * scale, (kernel, L, rho, np.max(np.abs(M @ M.T - S)) / scale)
    assert np.max(np.abs(off - mu)) <= 1e-10 * np.max(np.abs(mu)), (kernel, L, rho)


@pytest.fixture(scope="module")
def post_exe(tmp_path_factory):
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    exe = str(tmp_path_factory.mktemp("ss_post") / "ss_post_host_test")
    subprocess.run(["g++", "-O2", "-std=c++17", "-I", os.path.join(ROOT, "gpcc_b200", "csrc"),
                    os.path.join(ROOT, "tests", "host", "ss_post_host_test.cpp"), "-o", exe], check=True)
    return exe


def _spd(rng, D, scale):
    X = rng.standard_normal((D, D))
    return scale * (X @ X.T / D + 0.1 * np.eye(D))


@pytest.mark.parametrize("kernel", ["OU", "matern32", "matern52"])
def test_point_mean_weights(post_exe, kernel):
    """c1'm - w'lam equals the mean of ss::point_moments to 1e-13 relative, before the first step (dt1 = 0), between steps,
    after the last (no adjoint) and on a training time (dt1 = 0), for L = 1, 3, 8 and rho = 0.1, 300."""
    kid, d = {"OU": 0, "matern32": 2, "matern52": 3}[kernel], DIM[kernel]
    rng = np.random.default_rng(kid)
    cases, lines = [], []
    for L in (1, 3, 8):
        D = d + L
        iu = np.triu_indices(D)
        for rho in (0.1, 300.0):
            for dt1, later, dt2 in ((0.0, 1, 0.7), (0.4, 1, 0.2), (1.3, 0, 0.0), (0.0, 0, 0.0), (2e-3, 1, 5.0)):
                l = int(rng.integers(L))
                m, lam = rng.standard_normal(D), rng.standard_normal(D)
                P, Lam = _spd(rng, D, 1.0), _spd(rng, D, 0.5)
                head = "%d %d %d %.17g %.17g %.17g %d %.17g\n" % (kid, L, l, 0.5 + rng.random(), rho, dt1, later, dt2)
                body = " ".join("%.17g" % v for v in np.concatenate([m, P[iu]] + ([lam, Lam[iu]] if later else [])))
                lines.append(head + body + "\n")
                cases.append((L, rho, dt1, later))
    out = subprocess.run([post_exe], input="".join(lines), check=True, capture_output=True, text=True).stdout.split("\n")
    for line, case in zip(out, cases):
        mean, lin = (float(u) for u in line.split())
        assert abs(mean - lin) <= 1e-13 * max(1.0, abs(mean)), (kernel, case, mean, lin)
