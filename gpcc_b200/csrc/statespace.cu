// State-space method (gpcc_problem_set_method(p, GPCC_METHOD_STATESPACE)): the exact log-likelihood of the OU / Matérn
// models by a Kalman filter over the merged, delay-shifted times, in O(N (d+L)^2) per evaluation instead of the N^3 / 3 of
// the dense factorisation.
//
// Model: state x = [f-state (d); b (L)] in residual form (b has prior mean 0 and covariance diag(Sigma_b); the
// observations are resid = y - mu_b).  The f-block follows the kernel's SDE (ss_model.h), the b-block is static, and
// observation i of band l reads alpha_l x_0 + x_(d+l) with noise sigma_i^2.  The filter starts the f-block at P_inf,
// predicts the f-rows and f-columns over each gap and makes one rank-1 update per observation.  Its final b-block is the
// posterior of the shifts (postb, gpccfixdelay_marginaliseb.jl:248-252).
//
// Mapping: one group of G = (want_grad ? L+1 : 1) lanes per evaluation; lane j carries the primal and the forward-mode
// tangent of parameter j (alpha_1..alpha_L, rho), so no state is stored per step and lanes never communicate.  A group
// never straddles a warp.  Every lane of a group makes the same merge decisions (same data, same arithmetic), so the loop
// and its exit are uniform within the group.  Band-dependent parts are selects over an unrolled band loop: no register
// array is indexed dynamically.
//
// Data order: per band, a stable argsort of t (done once, when the method is switched on).  tau_l is constant within a
// band, so that order does not depend on the candidate; each evaluation merges the L sorted bands on the fly, taking
// the smallest t - tau_l, ties to the lowest band.  The merge is deterministic, so results are bitwise reproducible.
#include "gpcc_internal.h"
#include "kernfun.cuh"
#include "ss_model.h"

namespace gpcc {
namespace {

constexpr double LOG2PI = 1.8378770664093454836;

template <int D>
__host__ __device__ constexpr int sym(int i, int j) {      // packed upper triangle, row-major
    return i <= j ? i * D - i * (i - 1) / 2 + (j - i) : j * D - j * (j - 1) / 2 + (i - j);
}

struct Head { double t, r, s2; };

__device__ __forceinline__ Head load_point(const SSProblem& p, int i, int end, double tau) {
    Head h;
    if (i < end) { h.t = __ldg(p.t + i) - tau; h.r = __ldg(p.r + i); h.s2 = __ldg(p.s2 + i); }
    else { h.t = __builtin_huge_val(); h.r = 0.0; h.s2 = 1.0; }     // sentinel past the band's end: never taken
    return h;
}

template <int KID, int L, bool GRAD>
__global__ void __launch_bounds__(128) ss_filter_kernel(SSProblem p, int M, const double* __restrict__ delays,
                                                        const double* __restrict__ alpha, const double* __restrict__ rho,
                                                        double* ll_out, double* grad_out, int* info_out, double* postb) {
    constexpr int d = ss::Dim<KID>::d, D = d + L, NP = D * (D + 1) / 2;
    constexpr int G = GRAD ? L + 1 : 1, GPW = 32 / G;
    const int lane = threadIdx.x & 31;
    const int warp = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int grp = lane / G, j = lane - grp * G;
    const int e = warp * GPW + grp;
    if (grp >= GPW || e >= M) return;

    const double r_ho = rho[e];
    double al[L], tau[L];
#pragma unroll
    for (int l = 0; l < L; ++l) { al[l] = alpha[(size_t)e * L + l]; tau[l] = delays[(size_t)e * L + l]; }
    ss::Coef<d> c;
    ss::setup<KID>(r_ho, c);
    const bool trho = GRAD && j == L;        // this lane's tangent is d/drho (else d/dalpha_j)

    double m[D], P[NP], dm[D], dP[NP];
#pragma unroll
    for (int i = 0; i < D; ++i) { m[i] = 0.0; dm[i] = 0.0; }
#pragma unroll
    for (int i = 0; i < D; ++i)
#pragma unroll
        for (int k = i; k < D; ++k) {
            double v = 0.0, dv = 0.0;
            if (k < d) { v = c.Pinf[i][k]; dv = trho ? c.dPinf[i][k] : 0.0; }
            else if (i == k) v = p.Sigmab[i - d];
            P[sym<D>(i, k)] = v; dP[sym<D>(i, k)] = dv;
        }

    Head head[L], next[L];
    int pos[L];
    double prev = __builtin_huge_val();
#pragma unroll
    for (int l = 0; l < L; ++l) {
        const int a = p.band_start[l], b = p.band_start[l + 1];
        head[l] = load_point(p, a, b, tau[l]);
        next[l] = load_point(p, a + 1, b, tau[l]);
        pos[l] = a + 2;
        prev = fmin(prev, head[l].t);
    }

    double ll = 0.0, dll = 0.0;
    int info = 0;
    for (int step = 1; step <= p.N; ++step) {
        // ---- merge: smallest shifted time, ties to the lowest band ----
        int l = 0;
        double ts = head[0].t, r = head[0].r, s2 = head[0].s2, a = al[0];
#pragma unroll
        for (int lb = 1; lb < L; ++lb)
            if (head[lb].t < ts) { l = lb; ts = head[lb].t; r = head[lb].r; s2 = head[lb].s2; a = al[lb]; }
#pragma unroll
        for (int lb = 0; lb < L; ++lb)
            if (lb == l) { head[lb] = next[lb]; next[lb] = load_point(p, pos[lb], p.band_start[lb + 1], tau[lb]); ++pos[lb]; }
        const double Dt = ts - prev;
        prev = ts;

        // ---- predict the f-rows and f-columns over the gap (Dt == 0: A = I, Q = 0, nothing to do) ----
        if (Dt > 0.0) {
            double A[d][d], Q[d][d], dA[d][d], dQ[d][d];
            ss::step<KID, GRAD>(c, Dt, A, Q, dA, dQ);
            if (GRAD && !trho) {
#pragma unroll
                for (int i = 0; i < d; ++i)
#pragma unroll
                    for (int k = 0; k < d; ++k) { dA[i][k] = 0.0; dQ[i][k] = 0.0; }
            }
#pragma unroll
            for (int k = d; k < D; ++k) {               // P_fb = A P_fb, one column at a time
                double col[d], dcol[d];
#pragma unroll
                for (int i = 0; i < d; ++i) {
                    double s = 0.0, ds = 0.0;
#pragma unroll
                    for (int q = 0; q < d; ++q) {
                        s = fma(A[i][q], P[sym<D>(q, k)], s);
                        if (GRAD) ds = fma(dA[i][q], P[sym<D>(q, k)], fma(A[i][q], dP[sym<D>(q, k)], ds));
                    }
                    col[i] = s; dcol[i] = ds;
                }
#pragma unroll
                for (int i = 0; i < d; ++i) { P[sym<D>(i, k)] = col[i]; if (GRAD) dP[sym<D>(i, k)] = dcol[i]; }
            }
            double AP[d][d], dAP[d][d];      // A P_ff and its tangent
#pragma unroll
            for (int i = 0; i < d; ++i)
#pragma unroll
                for (int k = 0; k < d; ++k) {
                    double s = 0.0, ds = 0.0;
#pragma unroll
                    for (int q = 0; q < d; ++q) {
                        s = fma(A[i][q], P[sym<D>(q, k)], s);
                        if (GRAD) ds = fma(dA[i][q], P[sym<D>(q, k)], fma(A[i][q], dP[sym<D>(q, k)], ds));
                    }
                    AP[i][k] = s; dAP[i][k] = ds;
                }
#pragma unroll
            for (int i = 0; i < d; ++i) {
#pragma unroll
                for (int k = i; k < d; ++k) {           // P_ff = A P_ff A' + Q
                    double s = Q[i][k], ds = GRAD ? dQ[i][k] : 0.0;
#pragma unroll
                    for (int q = 0; q < d; ++q) {
                        s = fma(AP[i][q], A[k][q], s);
                        if (GRAD) ds = fma(dAP[i][q], A[k][q], fma(AP[i][q], dA[k][q], ds));
                    }
                    P[sym<D>(i, k)] = s;
                    if (GRAD) dP[sym<D>(i, k)] = ds;
                }
            }
            double mf[d], dmf[d];
#pragma unroll
            for (int i = 0; i < d; ++i) {
                double s = 0.0, ds = 0.0;
#pragma unroll
                for (int q = 0; q < d; ++q) {
                    s = fma(A[i][q], m[q], s);
                    if (GRAD) ds = fma(dA[i][q], m[q], fma(A[i][q], dm[q], ds));
                }
                mf[i] = s; dmf[i] = ds;
            }
#pragma unroll
            for (int i = 0; i < d; ++i) { m[i] = mf[i]; if (GRAD) dm[i] = dmf[i]; }
        }

        // ---- rank-1 update with h = a e_0 + e_(d+l) ----
        const double da = (GRAD && j == l) ? 1.0 : 0.0;        // d a / d(this lane's parameter)
        double Ph[D], dPh[D];
#pragma unroll
        for (int i = 0; i < D; ++i) {
            double s = 0.0, ds = 0.0;
#pragma unroll
            for (int lb = 0; lb < L; ++lb)
                if (lb == l) { s = P[sym<D>(i, d + lb)]; if (GRAD) ds = dP[sym<D>(i, d + lb)]; }
            Ph[i] = fma(a, P[sym<D>(i, 0)], s);
            if (GRAD) dPh[i] = fma(a, dP[sym<D>(i, 0)], fma(da, P[sym<D>(i, 0)], ds));
        }
        double Phb = 0.0, mb = 0.0, dPhb = 0.0, dmb = 0.0;
#pragma unroll
        for (int lb = 0; lb < L; ++lb)
            if (lb == l) { Phb = Ph[d + lb]; mb = m[d + lb]; if (GRAD) { dPhb = dPh[d + lb]; dmb = dm[d + lb]; } }
        const double S = fma(a, Ph[0], Phb) + s2;
        if (!(S > 0.0) || !(S < __builtin_huge_val())) { info = step; break; }
        const double v = r - fma(a, m[0], mb);
        const double iS = 1.0 / S;
        ll -= 0.5 * (LOG2PI + log(S) + v * v * iS);
        double k[D];
#pragma unroll
        for (int i = 0; i < D; ++i) k[i] = Ph[i] * iS;
        if (GRAD) {
            const double dS = fma(da, Ph[0], fma(a, dPh[0], dPhb));
            const double dv = -fma(da, m[0], fma(a, dm[0], dmb));
            dll -= 0.5 * (dS * iS + (2.0 * v * dv - v * v * dS * iS) * iS);
            double dk[D];
#pragma unroll
            for (int i = 0; i < D; ++i) dk[i] = (dPh[i] - k[i] * dS) * iS;
#pragma unroll
            for (int i = 0; i < D; ++i) dm[i] = fma(dk[i], v, fma(k[i], dv, dm[i]));
#pragma unroll
            for (int i = 0; i < D; ++i)
#pragma unroll
                for (int q = i; q < D; ++q) dP[sym<D>(i, q)] -= fma(dPh[i], k[q], Ph[i] * dk[q]);
        }
#pragma unroll
        for (int i = 0; i < D; ++i) m[i] = fma(k[i], v, m[i]);
#pragma unroll
        for (int i = 0; i < D; ++i)
#pragma unroll
            for (int q = i; q < D; ++q) P[sym<D>(i, q)] = fma(-Ph[i], k[q], P[sym<D>(i, q)]);
    }

    if (j == 0) {
        ll_out[e] = info ? -__builtin_huge_val() : ll;
        info_out[e] = info;
    }
    if (GRAD) grad_out[(size_t)e * (L + 1) + j] = info ? 0.0 : dll;
    if (postb && e == 0 && j == 0) {           // [L] mean, then [L][L] covariance (symmetric)
#pragma unroll
        for (int l = 0; l < L; ++l) {
            postb[l] = m[d + l] + p.mub[l];
#pragma unroll
            for (int q = 0; q < L; ++q) postb[L + l * L + q] = P[sym<D>(d + l, d + q)];
        }
    }
}

template <int KID, int L, bool GRAD>
cudaError_t launch_one(const SSProblem& p, const EvalBatch& b, double* postb, cudaStream_t stream) {
    constexpr int G = GRAD ? L + 1 : 1, GPW = 32 / G, THREADS = 128;
    const int warps = (b.M + GPW - 1) / GPW;
    const int blocks = (warps + THREADS / 32 - 1) / (THREADS / 32);
    ss_filter_kernel<KID, L, GRAD><<<blocks, THREADS, 0, stream>>>(p, b.M, b.delays, b.alpha, b.rho, b.ll, b.grad, b.info, postb);
    return cudaGetLastError();
}

template <int KID, int L>
cudaError_t launch_l(const SSProblem& p, const EvalBatch& b, double* postb, cudaStream_t stream) {
    if (p.L == L) return b.want_grad ? launch_one<KID, L, true>(p, b, postb, stream) : launch_one<KID, L, false>(p, b, postb, stream);
    if constexpr (L < MAX_BANDS) return launch_l<KID, L + 1>(p, b, postb, stream);
    return cudaErrorInvalidValue;
}

}  // namespace

cudaError_t statespace_launch(int kernel_id, const SSProblem& p, const EvalBatch& b, double* postb, cudaStream_t stream) {
    if (b.M <= 0) return cudaSuccess;
    switch (kernel_id) {
        case K_OU:  return launch_l<K_OU, 1>(p, b, postb, stream);
        case K_M32: return launch_l<K_M32, 1>(p, b, postb, stream);
        case K_M52: return launch_l<K_M52, 1>(p, b, postb, stream);
        default:       return cudaErrorInvalidValue;     // rbf: rejected by gpcc_problem_set_method
    }
}

}  // namespace gpcc
