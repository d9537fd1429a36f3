"""The O(N) draw of the state-space method (Problem.statespace_sample, gpcc_ss_sample) on the device: its exact covariance
against the dense oracle, impulse responses across the tiles of the scan up to N ~ 1e6, the generator and its
reproducibility, the argument checks, and delay recovery on data it drew."""
import ctypes as C
from types import SimpleNamespace

import numpy as np
import pytest
import scipy.linalg as sla

import gpcc_b200
from gpcc_b200 import Problem, _lib
from oracle import statespace as oss
from oracle.covariance import delayed_covariance
from ss_sample_reference import DIM, data

pytestmark = pytest.mark.gpu

TILE, SCAN = 64, 256          # merged steps per tile and threads of the aggregate scan (gpcc_b200/csrc/ss_sample.cu)
_dp = C.POINTER(C.c_double)


def _sobs(s):
    return np.concatenate([np.asarray(a, dtype=np.float64) ** 2 for a in s])


@pytest.mark.parametrize("kernel", ["OU", "matern32", "matern52"])
@pytest.mark.parametrize("L", [1, 2, 3, 8])
@pytest.mark.parametrize("rho", [0.1, 300.0])
def test_exact_covariance(ctx, kernel, L, rho):
    """z_in = the identity: the draws are the columns of the map M from deviates to f, and M M' = K + Sobs."""
    rng = np.random.default_rng(10 * L + int(rho))
    t, y, s, delays = data(rng, L)
    alpha = 0.6 + rng.random(L)
    p = Problem(t, y, s, kernel, ctx, method="statespace")
    S = DIM[kernel] + 1
    n = p.N * S
    f = p.statespace_sample(delays, alpha, rho, 0, nsamples=n, z=np.eye(n).reshape(n, p.N, S))
    ref = delayed_covariance(kernel, alpha, delays, rho, t) + np.diag(_sobs(s))
    err = np.max(np.abs(f.T @ f - ref))
    assert err <= 1e-10 * np.max(np.diag(ref)), (kernel, L, rho, err)


def _gap_bands(rng, n, span, gap_at, gap):
    """Two bands of sorted-then-shuffled times in [0, span + gap] with no time in (gap_at, gap_at + gap)."""
    out = []
    for m in n:
        u = np.sort(rng.uniform(0.0, span, m))
        out.append(rng.permutation(np.where(u > gap_at, u + gap, u)))
    return out


def _row0_expm(kernel, rho, tau, v):
    """[expm(F tau) v]_0 for many tau >= 0: F + lambda I is nilpotent, so expm(F tau) = exp(-lambda tau) sum_n (tau N)^n / n!
    (checked against scipy's expm at a few tau)."""
    F = oss.sde(kernel, rho)[0]
    d = F.shape[0]
    lam = -F[d - 1, d - 1] / d
    Nv = [v]
    for _ in range(1, d):
        Nv.append((F + lam * np.eye(d)) @ Nv[-1])

    def row0(x):
        return np.exp(-lam * x) * sum(x ** k / np.prod(np.arange(1, k + 1)) * Nv[k][0] for k in range(d))

    for x in (0.0, 0.37 / lam, 5.0 / lam):
        assert abs(row0(x) - (sla.expm(F * x) @ v)[0]) <= 1e-13 * max(1.0, np.abs(v).max())
    return row0(tau)


def _impulse_case(ctx, kernel, N, rho, span, seed):
    rng = np.random.default_rng(seed)
    n = [N // 2, N - N // 2]
    gap = 2.5 * rho                                              # lambda D >= 1 across the gap for every kernel
    t = _gap_bands(rng, n, span, 0.6 * span, gap)
    s = [0.1 + 0.05 * rng.random(m) for m in n]
    y = [np.sin(a) for a in t]
    delays, alpha = np.array([0.0, 1.3]), np.array([1.1, 0.7])
    p = Problem(t, y, s, kernel, ctx, method="statespace")
    pr = SimpleNamespace(t=t, L=2, N=p.N, band=np.repeat([0, 1], n))
    order, sh = oss.merge_order(pr, delays)
    d = DIM[kernel]
    S = d + 1
    i0 = order[0]
    k_gap = int(np.argmax(np.diff(sh[order]))) + 1              # first merged step after the gap
    ig = order[k_gap]
    Dg = sh[ig] - sh[order[k_gap - 1]]
    _, _, Pinf, _ = oss.sde(kernel, rho)
    Cg = np.linalg.cholesky(oss.transition(kernel, rho, Dg)[1])
    z = np.zeros((2 * d + 1, p.N, S))
    for c in range(d):
        z[c, i0, c] = 1.0                                        # process impulse e_c at the first merged point
        z[d + c, ig, c] = 1.0                                    # ... at the first point after the gap
    inoise = int(rng.integers(p.N))
    z[2 * d, inoise, d] = 1.0                                    # noise impulse
    f = p.statespace_sample(delays, alpha, rho, 0, nsamples=2 * d + 1, z=z)
    al = alpha[pr.band]
    cP = np.linalg.cholesky(Pinf)
    for c in range(d):
        ref = al * _row0_expm(kernel, rho, sh - sh[i0], cP[:, c])
        assert np.max(np.abs(f[c] - ref)) <= 1e-11 * alpha.max(), (kernel, N, c, np.max(np.abs(f[c] - ref)))
        after = sh >= sh[ig]
        after[order[:k_gap]] = False                             # ties with the gap step that precede it
        ref = np.where(after, al * _row0_expm(kernel, rho, np.maximum(sh - sh[ig], 0.0), Cg[:, c]), 0.0)
        assert np.max(np.abs(f[d + c] - ref)) <= 1e-11 * alpha.max(), (kernel, N, c, np.max(np.abs(f[d + c] - ref)))
    ref = np.zeros(p.N)
    ref[inoise] = np.concatenate(s)[inoise]
    assert np.array_equal(f[2 * d], ref)


@pytest.mark.parametrize("kernel", ["OU", "matern32", "matern52"])
@pytest.mark.parametrize("N", [TILE - 1, TILE, TILE + 1, 3 * TILE + 1])
def test_impulse_tile_edges(ctx, kernel, N):
    _impulse_case(ctx, kernel, N, rho=10.0, span=40.0, seed=N)


def test_impulse_tiles_overflow_one_scan_cta(ctx):
    N = 2 * TILE * SCAN + 37                                     # three chunks of the aggregate scan
    _impulse_case(ctx, "matern52", N, rho=20.0, span=200.0, seed=1)


def test_impulse_million_points(ctx):
    """N ~ 1e6 at rho = 300 over a span of 300: the response of the first point has not decayed at the last."""
    _impulse_case(ctx, "matern52", 1_000_003, rho=300.0, span=300.0, seed=2)


def _gen_problem(ctx, kernel="matern32", n=(400, 350, 300), seed=5):
    rng = np.random.default_rng(seed)
    t = [rng.uniform(0, 100, m) for m in n]
    s = [0.2 + 0.1 * rng.random(m) for m in n]
    return Problem(t, [np.cos(a) for a in t], s, kernel, ctx, method="statespace"), t, s


def test_generator_reproducible(ctx):
    p, _, _ = _gen_problem(ctx)
    d, a, r = np.array([0.0, 2.0, -3.0]), np.array([1.0, 1.5, 0.7]), 4.0
    f, z = p.statespace_sample(d, a, r, 7, nsamples=4, return_z=True)
    assert z.shape == (4, p.N, 3) and f.shape == (4, p.N)
    assert np.array_equal(f, p.statespace_sample(d, a, r, 7, nsamples=4))
    assert np.array_equal(f, p.statespace_sample(d, a, r, 123, nsamples=4, z=z))
    assert np.array_equal(f[:2], p.statespace_sample(d, a, r, 7, nsamples=2))
    g = p.statespace_sample(d, a, r, 8, nsamples=4)
    assert np.all(f != g)
    _, z2 = p.statespace_sample(d + np.array([0.0, 1.0, 2.5]), a, r, 7, nsamples=4, return_z=True)
    assert np.array_equal(z, z2)                                 # common random numbers across delays


def test_generator_moments(ctx):
    p, _, _ = _gen_problem(ctx, "matern52", (20000, 15000, 15000), 6)
    _, z = p.statespace_sample(np.zeros(3), np.ones(3), 3.0, 99, nsamples=5, return_z=True)
    x = z.ravel()
    n = x.size
    assert n >= 1_000_000
    assert abs(x.mean()) <= 5.0 / np.sqrt(n)
    assert abs(x.var() - 1.0) <= 5.0 * np.sqrt(2.0 / n)


def test_empirical_covariance(ctx):
    p, t, s = _gen_problem(ctx, "matern32", (40, 45, 35), 7)
    d, a, r = np.array([0.0, 5.0, -8.0]), np.array([1.2, 0.8, 1.5]), 6.0
    n = 20000
    f = p.statespace_sample(d, a, r, 2024, nsamples=n)
    Sig = delayed_covariance("matern32", a, d, r, t) + np.diag(_sobs(s))
    emp = f.T @ f / n
    se = np.sqrt((np.outer(np.diag(Sig), np.diag(Sig)) + Sig ** 2) / n)
    assert np.max(np.abs(emp - Sig) / se) <= 6.0


def test_errors(ctx):
    p, t, s = _gen_problem(ctx, "OU", (30, 20, 25), 8)
    lib = _lib.load()
    N = p.N
    d, a = np.zeros(3), np.ones(3)
    f = np.empty(N)

    def call(prob=p, dd=d, aa=a, rho=2.0, ns=1, z=None, out=f):
        return lib.gpcc_ss_sample(prob._h if prob is not None else None, dd.ctypes.data_as(_dp) if dd is not None else None,
                                  aa.ctypes.data_as(_dp), rho, 1, ns, z.ctypes.data_as(_dp) if z is not None else None,
                                  out.ctypes.data_as(_dp) if out is not None else None, None)

    assert call() == 0
    assert call(prob=None) == -1 and call(dd=None) == -1 and call(out=None) == -1
    assert call(aa=np.array([1.0, 0.0, 1.0])) == -2
    assert call(aa=np.array([1.0, np.nan, 1.0])) == -2
    assert call(dd=np.array([0.0, np.inf, 1.0])) == -3
    assert call(rho=0.0) == -4 and call(rho=np.nan) == -4
    assert call(ns=0) == -7
    z = np.zeros((1, N, 2))
    assert call(z=z) == 0
    z[0, N // 2, 1] = np.nan
    assert call(z=z) == -8
    dense = Problem(t, [np.cos(x) for x in t], s, "OU", ctx)
    assert call(prob=dense) == -5
    with pytest.raises(gpcc_b200.GpccError):
        p.statespace_sample(d, a, 2.0, 1, nsamples=2, z=np.zeros((1, N, 2)))
    with pytest.raises(gpcc_b200.GpccError):
        gpcc_b200.simulatedata_device(t, delays=d, alpha=a, b=np.zeros(3), kernel=gpcc_b200.rbf, ctx=ctx, method="statespace")


def test_abi():
    """gpcc_ss_sample is additive: the version stays 103 and callers look the symbol up."""
    lib = _lib.load()
    assert lib.gpcc_version() == 103
    assert hasattr(lib, "gpcc_ss_sample") and "gpcc_ss_sample" in _lib.EXPORTS


def test_delay_recovery_end_to_end(ctx):
    """Three Matern-3/2 bands of 4096 points drawn by simulatedata_device(method="statespace"); the state-space grid
    posterior over 41 delays of the third band peaks within one grid step of the true delay."""
    rng = np.random.default_rng(31)
    t = [np.sort(rng.uniform(0.0, 300.0, 4096)) for _ in range(3)]
    true = np.array([0.0, 2.0, 5.0])
    tt, y, s = gpcc_b200.simulatedata_device(t, delays=true, alpha=np.array([1.5, 1.2, 1.8]), b=np.array([3.0, -1.0, 0.5]),
                                             rho=5.0, kernel=gpcc_b200.matern32, seed=17, ctx=ctx, method="statespace")
    grid = np.linspace(3.0, 7.0, 41)
    cands = np.stack([np.zeros(41), np.full(41, 2.0), grid], 1)
    res = gpcc_b200.gpccgrid(tt, y, s, cands, kernel=gpcc_b200.matern32, iterations=1000, rhomax=20.0, ctx=ctx,
                             method="statespace")
    mode = grid[int(np.argmax(res["posterior"]))]
    assert abs(mode - true[2]) <= (grid[1] - grid[0]) + 1e-12, (mode, res["posterior"].max())
