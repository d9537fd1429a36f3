"""The O(N) draw of the state-space method without a GPU: the numpy route of tests/ss_sample_reference.py gives a linear map
M from the deviates to the draw whose M M' is K + Sobs of the dense oracle, and the step factor of
gpcc_b200/csrc/ss_model.h (ss::noise_factor, built with g++) factors the process noise of ss::step."""
import os
import shutil
import subprocess

import numpy as np
import pytest

import oracle
from oracle.covariance import delayed_covariance
from conftest import ROOT
from ss_sample_reference import DIM, data, sample_map


@pytest.mark.parametrize("kernel", ["OU", "matern32", "matern52"])
@pytest.mark.parametrize("L", [1, 2, 3, 8])
@pytest.mark.parametrize("rho", [0.1, 300.0])
def test_map_covariance_is_dense_covariance(kernel, L, rho):
    rng = np.random.default_rng(10 * L + int(rho))
    t, y, s, delays = data(rng, L)
    alpha = 0.6 + rng.random(L)
    pr = oracle.Problem(t, y, s, kernel)
    M = sample_map(pr, kernel, delays, alpha, rho)
    assert M.shape == (pr.N, pr.N * (DIM[kernel] + 1))
    ref = delayed_covariance(kernel, alpha, delays, rho, t) + np.diag(pr.sobs)
    err = np.max(np.abs(M @ M.T - ref))
    assert err <= 1e-10 * np.max(np.diag(ref)), (kernel, L, rho, err)


@pytest.fixture(scope="module")
def noise_exe(tmp_path_factory):
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    exe = str(tmp_path_factory.mktemp("ss_noise") / "ss_noise_host_test")
    subprocess.run(["g++", "-O2", "-std=c++17", "-I", os.path.join(ROOT, "gpcc_b200", "csrc"),
                    os.path.join(ROOT, "tests", "host", "ss_noise_host_test.cpp"), "-o", exe], check=True)
    return exe


@pytest.mark.parametrize("kernel", ["OU", "matern32", "matern52"])
def test_noise_factor(noise_exe, kernel):
    """Lower triangular with a non-negative diagonal, C C' = Q to 1e-14 relative to sqrt(Q_ii Q_jj), and C = 0 exactly at
    D = 0, over lambda D in {0, 1e-9, 1e-4, 1, 30}."""
    kid, d = {"OU": 0, "matern32": 2, "matern52": 3}[kernel], DIM[kernel]
    lam1 = {"OU": 1.0, "matern32": np.sqrt(3.0), "matern52": np.sqrt(5.0)}[kernel]    # lambda at rho = 1
    cases = [(rho, x) for rho in (0.1, 1.0, 300.0) for x in (0.0, 1e-9, 1e-4, 1.0, 30.0)]
    lines = "".join("%d %.17g %.17g\n" % (kid, rho, x * rho / lam1) for rho, x in cases)
    out = subprocess.run([noise_exe], input=lines, check=True, capture_output=True, text=True).stdout.strip().split("\n")
    assert len(out) == len(cases)
    for line, (rho, x) in zip(out, cases):
        v = np.array([float(u) for u in line.split()])
        Q, C = v[:d * d].reshape(d, d), v[d * d:].reshape(d, d)
        assert np.all(np.triu(C, 1) == 0.0) and np.all(np.diag(C) >= 0.0), (kernel, rho, x)
        if x == 0.0:
            assert np.all(Q == 0.0) and np.all(C == 0.0), (kernel, rho)
            continue
        sc = np.sqrt(np.outer(np.diag(Q), np.diag(Q)))
        assert np.all(np.diag(Q) > 0)
        assert np.max(np.abs(C @ C.T - Q) / sc) <= 1e-14, (kernel, rho, x, np.max(np.abs(C @ C.T - Q) / sc))
