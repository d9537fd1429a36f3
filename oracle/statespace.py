"""Kalman-filter route to the GPCC likelihood for the Markovian kernels (oracle; test infrastructure only).

For OU, matern32 and matern52 the model y_li = alpha_l f(t_li - tau_l) + b_l + eps_li is a linear-Gaussian state-space
model over the merged, delay-shifted times: state x = [f-state (d); b (L)], the f-block follows the kernel's SDE, the
b-block is static, observation i reads alpha_l x_0 + b_l.  A covariance-form filter over the N merged points gives the
same logL as the dense factorisation of K + Sobs + B, and its final b-block is postb (gpccfixdelay_marginaliseb.jl:248-252).

This is deliberately a different route from the device's closed forms (gpcc_b200/csrc/ss_model.h): the transition comes
from scipy.linalg.expm, the process noise from Q = P_inf - A P_inf A', and the rho-tangent of both from
scipy.linalg.expm_frechet.  Merge order: ascending shifted time, ties to the lowest band, then the input order.
"""
import numpy as np
import scipy.linalg as sla

from .model import LOG2PI

SQRT3, SQRT5 = np.sqrt(3.0), np.sqrt(5.0)


def sde(kernel, rho):
    """Drift F, stationary covariance P_inf and their rho-derivatives."""
    if kernel == "OU":
        lam, dlam = 1.0 / rho, -1.0 / rho ** 2
        F, dF = np.array([[-lam]]), np.array([[-dlam]])
        P, dP = np.array([[1.0]]), np.zeros((1, 1))
    elif kernel == "matern32":
        lam = SQRT3 / rho
        dlam = -lam / rho
        F = np.array([[0.0, 1.0], [-lam ** 2, -2 * lam]])
        dF = np.array([[0.0, 0.0], [-2 * lam, -2.0]]) * dlam
        P, dP = np.diag([1.0, lam ** 2]), np.diag([0.0, 2 * lam]) * dlam
    elif kernel == "matern52":
        lam = SQRT5 / rho
        dlam = -lam / rho
        F = np.array([[0.0, 1.0, 0.0], [0.0, 0.0, 1.0], [-lam ** 3, -3 * lam ** 2, -3 * lam]])
        dF = np.array([[0.0, 0.0, 0.0], [0.0, 0.0, 0.0], [-3 * lam ** 2, -6 * lam, -3.0]]) * dlam
        P = np.array([[1.0, 0.0, -lam ** 2 / 3], [0.0, lam ** 2 / 3, 0.0], [-lam ** 2 / 3, 0.0, lam ** 4]])
        dP = np.array([[0.0, 0.0, -2 * lam / 3], [0.0, 2 * lam / 3, 0.0], [-2 * lam / 3, 0.0, 4 * lam ** 3]]) * dlam
    else:
        raise ValueError(f"no finite state-space form for kernel {kernel!r}")
    return F, dF, P, dP


def transition(kernel, rho, dt):
    """A(dt), Q(dt) and their rho-derivatives."""
    F, dF, P, dP = sde(kernel, rho)
    A, dA = sla.expm_frechet(F * dt, dF * dt)
    Q = P - A @ P @ A.T
    dQ = dP - dA @ P @ A.T - A @ dP @ A.T - A @ P @ dA.T
    return A, Q, dA, dQ


def merge_order(problem, delays):
    s = np.concatenate([problem.t[l] - delays[l] for l in range(problem.L)])
    return np.lexsort((np.arange(problem.N), problem.band, s)), s


def filter(problem, kernel, delays, alpha, rho, want_grad=False):
    """(logL, grad or None, postb mean, postb covariance, info) of the filter.  grad = d logL / d(alpha_1..alpha_L, rho).
    info is the 1-based merged position of the first step with a non-positive or non-finite innovation variance."""
    pr = problem
    L = pr.L
    F, dF, Pinf, dPinf = sde(kernel, rho)
    d = F.shape[0]
    D = d + L
    order, s = merge_order(pr, delays)
    r = pr.Y - pr.mub[pr.band]
    m = np.zeros(D)
    P = np.zeros((D, D))
    P[:d, :d] = Pinf
    P[d:, d:] = np.diag(pr.Sigmab)
    nt = L + 1                                   # tangents: alpha_1..alpha_L, rho
    dm = np.zeros((nt, D))
    dP = np.zeros((nt, D, D))
    dP[L, :d, :d] = dPinf
    ll, g = 0.0, np.zeros(nt)
    prev = None
    for pos, i in enumerate(order):
        if prev is not None and s[i] != prev:
            A, Q, dA, dQ = transition(kernel, rho, s[i] - prev)
            dm[:, :d] = dm[:, :d] @ A.T
            dm[L, :d] += dA @ m[:d]
            m[:d] = A @ m[:d]
            T = np.zeros((D, D))
            T[:d, :d] = A
            T[d:, d:] = np.eye(L)
            dT = np.zeros((D, D))
            dT[:d, :d] = dA
            dP = np.einsum("ij,tjk,lk->til", T, dP, T)
            dP[L] += dT @ P @ T.T + T @ P @ dT.T
            dP[L, :d, :d] += dQ
            P = T @ P @ T.T
            P[:d, :d] += Q
        prev = s[i]
        l = pr.band[i]
        h = np.zeros(D)
        h[0], h[d + l] = alpha[l], 1.0
        dh = np.zeros((nt, D))
        dh[l, 0] = 1.0
        v = r[i] - h @ m
        Ph = P @ h
        S = h @ Ph + pr.sobs[i]
        if not (np.isfinite(S) and S > 0):
            return -np.inf, (np.zeros(nt) if want_grad else None), None, None, pos + 1
        dv = -(dh @ m) - dm @ h
        dPh = dP @ h + dh @ P
        dS = dh @ Ph + dPh @ h
        ll += -0.5 * (LOG2PI + np.log(S) + v * v / S)
        g += -0.5 * (dS / S + 2 * v * dv / S - v * v * dS / S ** 2)
        k = Ph / S
        dk = dPh / S - np.outer(dS, Ph) / S ** 2
        dm = dm + dk * v + np.outer(dv, k)
        m = m + k * v
        dP = dP - np.einsum("ti,j->tij", dPh, k) - np.einsum("i,tj->tij", Ph, dk)
        P = P - np.outer(Ph, k)
        P = 0.5 * (P + P.T)
        dP = 0.5 * (dP + dP.transpose(0, 2, 1))
    Sb = P[d:, d:]
    return ll, (g if want_grad else None), pr.mub + m[d:], 0.5 * (Sb + Sb.T), 0
