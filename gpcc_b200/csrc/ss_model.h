// State-space form of the three Markovian kernels of src/util.jl:15-52, for the Kalman filter of statespace.cu.
// Plain C++ behind GPCC_HD (like lbfgs.h), so that tests/test_statespace_cpu.py can build it with g++.
//
//   kernel     d   lambda      SDE state          k(tau)
//   OU         1   1/rho       f                  exp(-lambda tau)
//   matern32   2   sqrt3/rho   [f, f']            (1 + lambda tau) exp(-lambda tau)
//   matern52   3   sqrt5/rho   [f, f', f'']       (1 + lambda tau + (lambda tau)^2/3) exp(-lambda tau)
//
// The drift F has the d-fold eigenvalue -lambda, so N = F + lambda I is nilpotent and the transition is the finite sum
//   A(D) = exp(-lambda D) (I + D N + D^2 N^2 / 2)
// with no matrix exponential (transition_coef tabulates it).  The process noise is written as the integral it is,
//   Q(D) = q int_0^D g(s) g(s)' ds,   g(s) = A(s) e_{d-1} = exp(-lambda s) sum_a G[.][a] s^a,
// so that every entry is a short sum of I_n(D) = int_0^D s^n exp(-2 lambda s) ds, evaluated through a positive series
// of the regularised incomplete gamma function.  The difference P_inf - A P_inf A' would lose all digits when
// lambda D << 1 (dense sampling at rho = rhomax); it is used only from 2 lambda D = 4 on, where it loses less than one.
// D = 0 gives A = I and Q = 0 exactly.  All derivatives are with respect to rho.
#pragma once
#include <cmath>

#if defined(__CUDACC__)
#define GPCC_HD __host__ __device__
#define GPCC_HDFI __host__ __device__ __forceinline__
#else
#define GPCC_HD
#define GPCC_HDFI inline
#endif

namespace gpcc {
namespace ss {

template <int KID> struct Dim;                       // KID as in kernfun.cuh: 0 OU, 2 matern32, 3 matern52 (rbf has none)
template <> struct Dim<0> { static constexpr int d = 1; };
template <> struct Dim<2> { static constexpr int d = 2; };
template <> struct Dim<3> { static constexpr int d = 3; };

// Everything that depends on rho only: computed once per evaluation.
template <int d>
struct Coef {
    double lam, dlam;                 // lambda, d lambda / d rho = -lambda / rho
    double G[d][d], dG[d][d];         // g_i(s) = exp(-lambda s) sum_a G[i][a] s^a, and d/dlambda
    double q, dq;                     // spectral density of the driving noise, and d/dlambda
    double Pinf[d][d], dPinf[d][d];   // stationary covariance and d/drho
};

template <int KID>
GPCC_HD inline void setup(double rho, Coef<Dim<KID>::d>& c) {
    constexpr int d = Dim<KID>::d;
    for (int i = 0; i < d; ++i)
        for (int j = 0; j < d; ++j) { c.G[i][j] = c.dG[i][j] = c.Pinf[i][j] = c.dPinf[i][j] = 0.0; }
    if (KID == 0) {
        const double l = 1.0 / rho;
        c.lam = l;
        c.G[0][0] = 1.0;
        c.q = 2.0 * l; c.dq = 2.0;
        c.Pinf[0][0] = 1.0;
    } else if (KID == 2) {
        const double l = 1.7320508075688772935 / rho;
        c.lam = l;
        c.G[0][1] = 1.0;                                  // g0 = s
        c.G[1][0] = 1.0; c.G[1][1] = -l;                  // g1 = 1 - lambda s
        c.dG[1][1] = -1.0;
        c.q = 4.0 * l * l * l; c.dq = 12.0 * l * l;
        c.Pinf[0][0] = 1.0; c.Pinf[1][1] = l * l;
        c.dPinf[1][1] = 2.0 * l;
    } else {
        const double l = 2.2360679774997896964 / rho, l2 = l * l;
        c.lam = l;
        c.G[0][2] = 0.5;                                  // g0 = s^2/2
        c.G[1][1] = 1.0; c.G[1][2] = -0.5 * l;            // g1 = s - lambda s^2/2
        c.G[2][0] = 1.0; c.G[2][1] = -2.0 * l; c.G[2][2] = 0.5 * l2;   // g2 = 1 - 2 lambda s + lambda^2 s^2/2
        c.dG[1][2] = -0.5; c.dG[2][1] = -2.0; c.dG[2][2] = l;
        c.q = (16.0 / 3.0) * l2 * l2 * l; c.dq = (80.0 / 3.0) * l2 * l2;
        c.Pinf[0][0] = 1.0; c.Pinf[1][1] = l2 / 3.0; c.Pinf[2][2] = l2 * l2;
        c.Pinf[0][2] = c.Pinf[2][0] = -l2 / 3.0;
        c.dPinf[1][1] = 2.0 * l / 3.0; c.dPinf[2][2] = 4.0 * l2 * l;
        c.dPinf[0][2] = c.dPinf[2][0] = -2.0 * l / 3.0;
    }
    c.dlam = -c.lam / rho;
    for (int i = 0; i < d; ++i)
        for (int j = 0; j < d; ++j) c.dPinf[i][j] *= c.dlam;
}

// I_n(D) = int_0^D s^n exp(-2 lambda s) ds for n = 0..NI-1, for u = 2 lambda D < 4.  With the regularised incomplete gamma
// P(n+1, u) = exp(-u) sum_{k > n} u^k / k!:  I_n = n! / (2 lambda)^(n+1) P(n+1, u).  The top order comes from its positive
// series (30 terms reach 1e-19 relative below u = 4) and the lower ones from P(n, u) = P(n+1, u) + exp(-u) u^n / n!,
// which adds positive terms only.  u = 0 gives I = 0 exactly.
template <int NI>
GPCC_HD inline void incgamma_moments(double lam, double u, double* I) {
    const double eu = exp(-u);
    double tk[NI + 1];                    // u^k / k!
    tk[0] = 1.0;
    for (int k = 1; k <= NI; ++k) tk[k] = tk[k - 1] * (u / k);
    double s = 0.0, t = tk[NI];
    for (int j = 1; j <= 30; ++j) { t *= u / (NI + j); s += t; }
    double P = eu * (tk[NI] + s);         // P(NI, u), then downwards
    const double r = 1.0 / (2.0 * lam);
    double f = r;                         // n! r^(n+1)
    for (int n = 1; n < NI; ++n) f *= n * r;
    for (int n = NI - 1; n >= 0; --n) {
        I[n] = f * P;
        if (n > 0) { P += eu * tk[n]; f /= n * r; }
    }
}

// Coefficient k of the polynomial p_ij of A(D) = exp(-x) (I + D N + D^2 N^2 / 2), x = lambda D (see step()).
GPCC_HD constexpr double transition_coef(int kid, int i, int j, int k) {
    const double ou[1][1][3] = {{{1, 0, 0}}};
    const double m32[2][2][3] = {{{1, 1, 0}, {1, 0, 0}},
                                 {{0, -1, 0}, {1, -1, 0}}};
    const double m52[3][3][3] = {{{1, 1, 0.5}, {1, 1, 0}, {0.5, 0, 0}},
                                 {{0, 0, -0.5}, {1, 1, -1}, {1, -0.5, 0}},
                                 {{0, -1, 0.5}, {0, -3, 1}, {1, -2, 0.5}}};
    return kid == 0 ? ou[0][0][k] : kid == 2 ? m32[i][j][k] : m52[i][j][k];
}

// Transition and process noise over a step D >= 0, and their rho-derivatives (dA, dQ may be skipped with want_d = false).
template <int KID, bool want_d>
GPCC_HD inline void step(const Coef<Dim<KID>::d>& c, double D, double (&A)[Dim<KID>::d][Dim<KID>::d],
                         double (&Q)[Dim<KID>::d][Dim<KID>::d], double (&dA)[Dim<KID>::d][Dim<KID>::d],
                         double (&dQ)[Dim<KID>::d][Dim<KID>::d]) {
    constexpr int d = Dim<KID>::d, NI = 2 * d;
    const double x = c.lam * D, e = exp(-x);
    // A_ij = e s_ij p_ij(x), s_ij = D^(j-i) above the diagonal and lambda^(i-j) below.  With x = lambda D the lambda-
    // derivative is e s_ij D (p' - p)(x) above (and on) the diagonal and e lambda^(i-j-1) (x (p' - p) + (i-j) p)(x) below;
    // the coefficients of p' - p are formed exactly, so that the cancellation of p' against p costs nothing at small x.
    for (int i = 0; i < d; ++i)
        for (int j = 0; j < d; ++j) {
            const double a0 = transition_coef(KID, i, j, 0), a1 = transition_coef(KID, i, j, 1), a2 = transition_coef(KID, i, j, 2);
            const double pv = a0 + x * (a1 + x * a2);
            const double qv = (a1 - a0) + x * ((2.0 * a2 - a1) + x * (-a2));     // p' - p
            double sc = 1.0, dsc;
            if (j >= i) {
                for (int k = i; k < j; ++k) sc *= D;
                dsc = sc * D * qv;
            } else {
                double lp = 1.0;                          // lambda^(i-j-1)
                for (int k = j + 1; k < i; ++k) lp *= c.lam;
                sc = lp * c.lam;
                dsc = lp * (x * qv + (i - j) * pv);
            }
            A[i][j] = e * sc * pv;
            if (want_d) dA[i][j] = c.dlam * e * dsc;
        }
    const double u = 2.0 * c.lam * D;
    if (u < 4.0) {
        // Q_ij = q sum_ab G_ia G_jb I_(a+b);  dI_n/dlambda = -2 I_(n+1)
        double I[NI];
        incgamma_moments<NI>(c.lam, u, I);
        for (int i = 0; i < d; ++i)
            for (int j = i; j < d; ++j) {
                double s = 0.0, ds = 0.0;
                for (int a = 0; a < d; ++a)
                    for (int b = 0; b < d; ++b) {
                        const double gg = c.G[i][a] * c.G[j][b];
                        s += gg * I[a + b];
                        if (want_d) ds += (c.dG[i][a] * c.G[j][b] + c.G[i][a] * c.dG[j][b]) * I[a + b] - 2.0 * gg * I[a + b + 1];
                    }
                Q[i][j] = Q[j][i] = c.q * s;
                if (want_d) dQ[i][j] = dQ[j][i] = c.dlam * (c.dq * s + c.q * ds);
            }
    } else {
        // A P_inf A' is at most ~0.7 of P_inf here: the difference loses under one digit, and its derivative is the small
        // term it is instead of the cancelling sum above
        double AP[d][d], dAP[d][d];
        for (int i = 0; i < d; ++i)
            for (int j = 0; j < d; ++j) {
                double s = 0.0, ds = 0.0;
                for (int k = 0; k < d; ++k) {
                    s += A[i][k] * c.Pinf[k][j];
                    if (want_d) ds += dA[i][k] * c.Pinf[k][j] + A[i][k] * c.dPinf[k][j];
                }
                AP[i][j] = s; dAP[i][j] = ds;
            }
        for (int i = 0; i < d; ++i)
            for (int j = i; j < d; ++j) {
                double s = 0.0, ds = 0.0;
                for (int k = 0; k < d; ++k) {
                    s += AP[i][k] * A[j][k];
                    if (want_d) ds += dAP[i][k] * A[j][k] + AP[i][k] * dA[j][k];
                }
                Q[i][j] = Q[j][i] = c.Pinf[i][j] - s;
                if (want_d) dQ[i][j] = dQ[j][i] = c.dPinf[i][j] - ds;
            }
    }
}

// Lower Cholesky factor C (C C' = Q, upper part zero) of a process noise or stationary covariance (the sampler of
// ss_sample.cu).  Q's entries span many orders of magnitude at small lambda D (Q_ij ~ D^(2d-1-i-j)), so Q is factored in
// diagonally scaled form, Q = S R S with S = diag(sqrt(Q_ii)) and R the correlation matrix, C = S chol(R): its rounding
// error is relative to sqrt(Q_ii Q_jj) entry by entry.  A zero diagonal entry or a non-positive pivot (rounding) gives a
// zero column, so D = 0 (Q = 0 exactly) gives C = 0 exactly.
template <int d>
GPCC_HD inline void noise_factor(const double (&Q)[d][d], double (&C)[d][d]) {
    double s[d];
    for (int i = 0; i < d; ++i) s[i] = Q[i][i] > 0.0 ? sqrt(Q[i][i]) : 0.0;
    for (int i = 0; i < d; ++i)
        for (int j = 0; j < d; ++j) C[i][j] = 0.0;
    for (int j = 0; j < d; ++j) {                 // column j of chol(R), then scaled by S
        if (!(s[j] > 0.0)) continue;
        double p = 1.0;
        for (int k = 0; k < j; ++k) p -= C[j][k] * C[j][k];
        if (!(p > 0.0)) continue;
        const double cjj = sqrt(p);
        C[j][j] = cjj;
        for (int i = j + 1; i < d; ++i) {
            if (!(s[i] > 0.0)) continue;
            double r = Q[i][j] / (s[i] * s[j]);
            for (int k = 0; k < j; ++k) r -= C[i][k] * C[j][k];
            C[i][j] = r / cjj;
        }
    }
    for (int i = 0; i < d; ++i)
        for (int j = 0; j <= i; ++j) C[i][j] *= s[i];
}

template <int D>
GPCC_HD constexpr int sym(int i, int j) {      // packed upper triangle, row-major
    return i <= j ? i * D - i * (i - 1) / 2 + (j - i) : j * D - j * (j - 1) / 2 + (i - j);
}

// Moments of x = [f-state (d); b (D - d)] carried over a gap with the f-block transition A and process noise Q (the b-block
// is static): m_f = A m_f, P_fb = A P_fb, P_ff = A P_ff A' + Q.  The primal lines of the gap predict of ss_filter_kernel
// (statespace.cu), which keeps its own inline copy: called from there, a shared function changes the register allocation
// and the spills of eight gradient instantiations of that kernel.
template <int d, int D>
GPCC_HDFI void predict_moments(const double (&A)[d][d], const double (&Q)[d][d], double (&m)[D], double (&P)[D * (D + 1) / 2]) {
#pragma unroll
    for (int k = d; k < D; ++k) {               // P_fb = A P_fb, one column at a time
        double col[d];
#pragma unroll
        for (int i = 0; i < d; ++i) {
            double s = 0.0;
#pragma unroll
            for (int q = 0; q < d; ++q) s = fma(A[i][q], P[sym<D>(q, k)], s);
            col[i] = s;
        }
#pragma unroll
        for (int i = 0; i < d; ++i) P[sym<D>(i, k)] = col[i];
    }
    double AP[d][d];                            // A P_ff
#pragma unroll
    for (int i = 0; i < d; ++i)
#pragma unroll
        for (int k = 0; k < d; ++k) {
            double s = 0.0;
#pragma unroll
            for (int q = 0; q < d; ++q) s = fma(A[i][q], P[sym<D>(q, k)], s);
            AP[i][k] = s;
        }
#pragma unroll
    for (int i = 0; i < d; ++i)
#pragma unroll
        for (int k = i; k < d; ++k) {           // P_ff = A P_ff A' + Q
            double s = Q[i][k];
#pragma unroll
            for (int q = 0; q < d; ++q) s = fma(AP[i][q], A[k][q], s);
            P[sym<D>(i, k)] = s;
        }
    double mf[d];
#pragma unroll
    for (int i = 0; i < d; ++i) {
        double s = 0.0;
#pragma unroll
        for (int q = 0; q < d; ++q) s = fma(A[i][q], m[q], s);
        mf[i] = s;
    }
#pragma unroll
    for (int i = 0; i < d; ++i) m[i] = mf[i];
}

// Smoothed mean and variance of h'x, h = a e_0 + e_(d+l), at a test time t between two training steps (statespace.cu, the
// fit state).  On entry m, P are the filtered moments of the last training step i at or before t (the prior if t precedes
// every training point); dt1 = t - s_i.  lam, Lam (packed) are the Bryson-Frazier adjoint of step i+1 before its update,
// so that the smoothed moments there are m- - P- lam and P- - P- Lam P-; NULL when t follows the last training step.
// dt2 = s_(i+1) - t > 0.  At t the adjoint is A2' lam and A2' Lam A2 (A2 over dt2, identity on the b-block), hence with
// u = P h and w = A2 u:  mean = h'm - w'lam,  var = h'P h - w' Lam w.  No matrix is inverted.
template <int KID, int L>
GPCC_HD inline void point_moments(const Coef<Dim<KID>::d>& c, int l, double a, double (&m)[Dim<KID>::d + L],
                                  double (&P)[(Dim<KID>::d + L) * (Dim<KID>::d + L + 1) / 2], double dt1,
                                  const double* lam, const double* Lam, double dt2, double& mean, double& var) {
    constexpr int d = Dim<KID>::d, D = d + L;
    double A[d][d], Q[d][d], dA[d][d], dQ[d][d];
    if (dt1 > 0.0) {
        step<KID, false>(c, dt1, A, Q, dA, dQ);
        predict_moments<d, D>(A, Q, m, P);
    }
    double u[D];
    for (int i = 0; i < D; ++i) u[i] = fma(a, P[sym<D>(i, 0)], P[sym<D>(i, d + l)]);
    mean = fma(a, m[0], m[d + l]);
    var = fma(a, u[0], u[d + l]);
    if (!lam) return;
    step<KID, false>(c, dt2, A, Q, dA, dQ);
    double w[D];
    for (int i = 0; i < D; ++i) {
        double s = i < d ? 0.0 : u[i];
        if (i < d)
            for (int q = 0; q < d; ++q) s = fma(A[i][q], u[q], s);
        w[i] = s;
    }
    double wl = 0.0, wLw = 0.0;
    for (int i = 0; i < D; ++i) {
        wl = fma(w[i], lam[i], wl);
        double s = 0.0;
        for (int q = 0; q < D; ++q) s = fma(Lam[sym<D>(i, q)], w[q], s);
        wLw = fma(w[i], s, wLw);
    }
    mean -= wl;
    var -= wLw;
}

// The mean of point_moments as a linear function of the data, for the posterior draws of ss_post_sample.cu: with m and lam
// as there (m the filtered mean of step i, lam the adjoint of step i+1; neither is read here), mean = c1'm - w'lam, where
// c1 = T1'h (T1: A over dt1 on the f-block, identity on the b-block) and w = T2 P1 h (P1: P predicted over dt1, T2: A over
// dt2); w = 0 when later is false.  c1 and w depend on the covariances only, so one pair serves every sample.  P is
// overwritten with P1.
template <int KID, int L>
GPCC_HD inline void point_mean_weights(const Coef<Dim<KID>::d>& c, int l, double a,
                                       double (&P)[(Dim<KID>::d + L) * (Dim<KID>::d + L + 1) / 2], double dt1, bool later,
                                       double dt2, double (&c1)[Dim<KID>::d + L], double (&w)[Dim<KID>::d + L]) {
    constexpr int d = Dim<KID>::d, D = d + L;
    double A[d][d], Q[d][d], dA[d][d], dQ[d][d];
    for (int i = 0; i < D; ++i) c1[i] = i < d ? (i == 0 ? a : 0.0) : (i == d + l ? 1.0 : 0.0);
    if (dt1 > 0.0) {
        step<KID, false>(c, dt1, A, Q, dA, dQ);
        double m0[D];
        for (int i = 0; i < D; ++i) m0[i] = 0.0;
        predict_moments<d, D>(A, Q, m0, P);
        for (int i = 0; i < d; ++i) c1[i] = a * A[0][i];
    }
    double u[D];
    for (int i = 0; i < D; ++i) u[i] = fma(a, P[sym<D>(i, 0)], P[sym<D>(i, d + l)]);
    for (int i = 0; i < D; ++i) w[i] = 0.0;
    if (!later) return;
    step<KID, false>(c, dt2, A, Q, dA, dQ);
    for (int i = 0; i < D; ++i) {
        double s = i < d ? 0.0 : u[i];
        if (i < d)
            for (int q = 0; q < d; ++q) s = fma(A[i][q], u[q], s);
        w[i] = s;
    }
}

}  // namespace ss
}  // namespace gpcc
