"""The state-space method without a GPU: the Kalman-filter oracle (oracle/statespace.py) against the dense oracle on every
OU / Matérn golden fixture and on edge cases, and the closed forms of gpcc_b200/csrc/ss_model.h (built with g++) against
the matrix exponential evaluated at 80 digits."""
import os
import shutil
import subprocess

import mpmath
import numpy as np
import pytest

import oracle
from oracle import statespace as ss
from conftest import load_golden, ROOT

FIXTURES = ["loglik_2band_OU", "loglik_2band_matern32", "loglik_2band_matern52", "loglik_3band_OU",
            "loglik_3band_matern32", "loglik_3band_matern52", "loglik_ragged_OU", "loglik_3x64_matern52"]


def _rel(a, b):
    return np.max(np.abs(np.asarray(a) - np.asarray(b))) / np.max(np.abs(np.asarray(b)))


@pytest.mark.parametrize("name", FIXTURES)
def test_filter_matches_dense_oracle_on_golden_rows(name):
    g = load_golden(name)
    pr = oracle.Problem(g["tb"], g["yb"], g["sb"], g["kernel"])
    for j in range(len(g["rho"])):
        ll, grad, mu, S, info = ss.filter(pr, g["kernel"], g["delays"][j], g["alpha"][j], g["rho"][j], want_grad=True)
        assert info == 0
        assert abs(ll - g["loglik"][j]) <= 1e-12 * abs(g["loglik"][j]), (name, j)
        assert _rel(grad, g["grad"][j]) <= 1e-9, (name, j)
        mu_r, S_r = pr.postb(g["delays"][j], g["alpha"][j], g["rho"][j])
        assert _rel(mu, mu_r) <= 1e-12 and _rel(S, S_r) <= 1e-12, (name, j)


def _edge_problem(case, rng):
    """Data for the edge cases: unsorted times, duplicates inside a band, coinciding shifted times, L = 1 and 8, a band
    of two points."""
    if case == "unsorted":
        t = [rng.permutation(np.sort(rng.uniform(0, 30, n))) for n in (25, 30, 20)]
        delays = np.array([0.0, 2.5, 4.0])
    elif case == "duplicates":
        base = [np.sort(rng.uniform(0, 30, n)) for n in (20, 24)]
        t = [np.concatenate([b, b[::3]]) for b in base]
        delays = np.array([0.0, 1.5])
    elif case == "coincident":
        t0 = np.sort(rng.uniform(0, 30, 30))
        t = [t0, t0 + 3.0, t0[:15] + 5.0]
        delays = np.array([0.0, 3.0, 5.0])
    elif case == "L1":
        t = [np.sort(rng.uniform(0, 30, 40))]
        delays = np.array([0.0])
    elif case == "L8":
        t = [np.sort(rng.uniform(0, 30, 12)) for _ in range(8)]
        delays = np.linspace(0.0, 7.0, 8)
    else:                                           # "two_points"
        t = [np.sort(rng.uniform(0, 30, 30)), np.array([4.0, 11.0])]
        delays = np.array([0.0, 1.0])
    y = [np.sin(a / 3.0) + 0.3 * rng.standard_normal(len(a)) for a in t]
    s = [0.2 + 0.1 * rng.random(len(a)) for a in t]
    alpha = 0.8 + 0.8 * rng.random(len(t))
    return t, y, s, delays, alpha


EDGE = ["unsorted", "duplicates", "coincident", "L1", "L8", "two_points"]


@pytest.mark.parametrize("kernel", ["OU", "matern32", "matern52"])
@pytest.mark.parametrize("case", EDGE)
@pytest.mark.parametrize("rho", [0.1, 300.0])
def test_filter_edge_cases(kernel, case, rho):
    t, y, s, delays, alpha = _edge_problem(case, np.random.default_rng(EDGE.index(case)))
    pr = oracle.Problem(t, y, s, kernel)
    ll, grad, mu, S, info = ss.filter(pr, kernel, delays, alpha, rho, want_grad=True)
    rl, rg = pr.loglik_grad(delays, alpha, rho)
    mu_r, S_r = pr.postb(delays, alpha, rho)
    assert info == 0
    assert abs(ll - rl) <= 1e-10 * abs(rl)
    assert _rel(grad, rg) <= 1e-7
    assert _rel(mu, mu_r) <= 1e-10 and _rel(S, S_r) <= 1e-10


# ---- closed forms of ss_model.h ---------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def model_exe(tmp_path_factory):
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    exe = str(tmp_path_factory.mktemp("ss_model") / "ss_model_host_test")
    subprocess.run(["g++", "-O2", "-std=c++17", "-I", os.path.join(ROOT, "gpcc_b200", "csrc"),
                    os.path.join(ROOT, "tests", "host", "ss_model_host_test.cpp"), "-o", exe], check=True)
    return exe


def _mp_reference(kernel, rho, dt):
    """A, Q = P_inf - A P_inf A' and their rho-derivatives (Fréchet derivative of expm by the block-triangular
    exponential) at 80 digits, where the cancellation in Q costs nothing."""
    mpmath.mp.dps = 80
    rho = mpmath.mpf(rho)
    dt = mpmath.mpf(dt)
    if kernel == "OU":
        lam = 1 / rho
        F = mpmath.matrix([[-lam]]); dF = mpmath.matrix([[1 / rho ** 2]])
        P = mpmath.matrix([[1]]); dP = mpmath.matrix([[0]])
    elif kernel == "matern32":
        lam = mpmath.sqrt(3) / rho; dl = -lam / rho
        F = mpmath.matrix([[0, 1], [-lam ** 2, -2 * lam]]); dF = mpmath.matrix([[0, 0], [-2 * lam * dl, -2 * dl]])
        P = mpmath.matrix([[1, 0], [0, lam ** 2]]); dP = mpmath.matrix([[0, 0], [0, 2 * lam * dl]])
    else:
        lam = mpmath.sqrt(5) / rho; dl = -lam / rho
        F = mpmath.matrix([[0, 1, 0], [0, 0, 1], [-lam ** 3, -3 * lam ** 2, -3 * lam]])
        dF = mpmath.matrix([[0, 0, 0], [0, 0, 0], [-3 * lam ** 2 * dl, -6 * lam * dl, -3 * dl]])
        P = mpmath.matrix([[1, 0, -lam ** 2 / 3], [0, lam ** 2 / 3, 0], [-lam ** 2 / 3, 0, lam ** 4]])
        dP = mpmath.matrix([[0, 0, -2 * lam * dl / 3], [0, 2 * lam * dl / 3, 0], [-2 * lam * dl / 3, 0, 4 * lam ** 3 * dl]])
    d = F.rows
    B = mpmath.zeros(2 * d, 2 * d)
    for i in range(d):
        for j in range(d):
            B[i, j] = B[d + i, d + j] = F[i, j] * dt
            B[i, d + j] = dF[i, j] * dt
    E = mpmath.expm(B)
    A = E[0:d, 0:d]
    dA = E[0:d, d:2 * d]
    Q = P - A * P * A.T
    dQ = dP - dA * P * A.T - A * dP * A.T - A * P * dA.T
    return [np.array([[float(M[i, j]) for j in range(d)] for i in range(d)]) for M in (A, Q, dA, dQ)]


LAMBDA = {"OU": 1.0, "matern32": np.sqrt(3.0), "matern52": np.sqrt(5.0)}
KID = {"OU": 0, "matern32": 2, "matern52": 3}


@pytest.mark.parametrize("kernel", ["OU", "matern32", "matern52"])
def test_closed_forms_against_matrix_exponential(model_exe, kernel):
    cases = [(rho, x * rho / LAMBDA[kernel]) for rho in (0.1, 3.5, 300.0) for x in (0.0, 1e-9, 1e-4, 1.0, 30.0)]
    inp = "".join("%d %.17g %.17g\n" % (KID[kernel], rho, dt) for rho, dt in cases)
    out = subprocess.run([model_exe], input=inp, check=True, capture_output=True, text=True).stdout.splitlines()
    assert len(out) == len(cases)
    for (rho, dt), line in zip(cases, out):
        v = np.array([float(x) for x in line.split()])
        d = int(round(np.sqrt(len(v) / 4)))
        A, Q, dA, dQ = v.reshape(4, d, d)
        rA, rQ, rdA, rdQ = _mp_reference(kernel, rho, dt)
        where = (kernel, rho, dt)
        if dt == 0.0:
            assert np.array_equal(A, np.eye(d)) and np.all(Q == 0.0) and np.all(dA == 0.0) and np.all(dQ == 0.0), where
            continue
        # every entry relative to itself, up to rounding against its natural scale: for A_ij = e^-x s_ij p_ij(x)
        # (s_ij = dt^(j-i) above the diagonal, lambda^(i-j) below) that is e^-x s_ij (1 + x + x^2), so that an entry at a
        # root of p_ij, such as (1 - x) e^-x at x = 1, is held to rounding; likewise for dA.  For Q and dQ it is the
        # geometric mean of the two diagonal entries (the off-diagonal covariances at x = 30 are ~e^-60 of the diagonal).
        lam = LAMBDA[kernel] / rho
        x = lam * dt
        i, j = np.indices((d, d))
        s = np.where(j >= i, dt ** np.maximum(j - i, 0), lam ** np.maximum(i - j, 0))
        nat_A = np.exp(-x) * s * (1 + x + x * x)
        nat_dA = (lam / rho) * np.exp(-x) * (s / lam) * np.where(j >= i, x, 1.0) * (1 + x + x * x + x ** 3)
        for M, R, nat in ((A, rA, nat_A), (Q, rQ, None), (dA, rdA, nat_dA), (dQ, rdQ, None)):
            if nat is None:
                nat = np.sqrt(np.outer(np.abs(np.diag(R)), np.abs(np.diag(R))))
            assert np.all(np.abs(M - R) <= 1e-13 * np.abs(R) + 1e-15 * nat), (where, M, R)
