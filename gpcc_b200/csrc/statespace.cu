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

using ss::sym;

struct Head { double t, r, s2; };

__device__ __forceinline__ Head load_point(const SSProblem& p, int i, int end, double tau) {
    Head h;
    if (i < end) { h.t = __ldg(p.t + i) - tau; h.r = __ldg(p.r + i); h.s2 = __ldg(p.s2 + i); }
    else { h.t = __builtin_huge_val(); h.r = 0.0; h.s2 = 1.0; }     // sentinel past the band's end: never taken
    return h;
}

// STORE (with GRAD = false and M = 1; the fit state of gpcc_ss_state_create): also writes, per merged step, the shifted time,
// the band and the filtered moments after the update to `st`.
template <int KID, int L, bool GRAD, bool STORE = false>
__global__ void __launch_bounds__(128) ss_filter_kernel(SSProblem p, int M, const double* __restrict__ delays,
                                                        const double* __restrict__ alpha, const double* __restrict__ rho,
                                                        double* ll_out, double* grad_out, int* info_out, double* postb,
                                                        SSStore st) {
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
        if (STORE) {
            const size_t o = (size_t)(step - 1);
            st.t[o] = ts;
            st.band[o] = l;
#pragma unroll
            for (int i = 0; i < D; ++i) st.m[o * D + i] = m[i];
#pragma unroll
            for (int i = 0; i < NP; ++i) st.P[o * NP + i] = P[i];
        }
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
    ss_filter_kernel<KID, L, GRAD><<<blocks, THREADS, 0, stream>>>(p, b.M, b.delays, b.alpha, b.rho, b.ll, b.grad, b.info, postb, SSStore{});
    return cudaGetLastError();
}

template <int KID, int L>
cudaError_t launch_l(const SSProblem& p, const EvalBatch& b, double* postb, cudaStream_t stream) {
    if (p.L == L) return b.want_grad ? launch_one<KID, L, true>(p, b, postb, stream) : launch_one<KID, L, false>(p, b, postb, stream);
    if constexpr (L < MAX_BANDS) return launch_l<KID, L + 1>(p, b, postb, stream);
    return cudaErrorInvalidValue;
}

// ---- fit state of the state-space method (gpcc_ss_state_*): stored forward pass, backward pass, per-point predictions ----
constexpr double JITTER = 1e-8;       // added to every predictive variance, as the dense fit state does (predict.cu)
constexpr double SIGMA_FLOOR = 1e-6;  // sd = sqrt(max(var + JITTER, SIGMA_FLOOR)), as the dense fit state does

template <int KID, int L>
__device__ __forceinline__ void prior_moments(const ss::Coef<ss::Dim<KID>::d>& c, const SSProblem& p,
                                              double (&m)[ss::Dim<KID>::d + L],
                                              double (&P)[(ss::Dim<KID>::d + L) * (ss::Dim<KID>::d + L + 1) / 2]) {
    constexpr int d = ss::Dim<KID>::d, D = d + L;
#pragma unroll
    for (int i = 0; i < D; ++i) {
        m[i] = 0.0;
#pragma unroll
        for (int k = i; k < D; ++k) P[sym<D>(i, k)] = k < d ? c.Pinf[i][k] : i == k ? p.Sigmab[i - d] : 0.0;
    }
}

// Bryson-Frazier backward pass over the stored forward pass: one thread, the steps are one sequential chain.  The predicted
// moments of step k are recomputed from the stored filtered moments of step k-1 with the filter's own predict, so gain and
// innovation are those of the forward pass.  With lam^, Lam^ the adjoint after the update of step k (zero after the last),
// k = P- h / S and w = Lam^ k, the adjoint before the update is
//   lam~ = (I - k h')' lam^ - h v / S             = lam^ - h (k'lam^ + v / S)
//   Lam~ = (I - k h')' Lam^ (I - k h') + h h' / S = Lam^ - h w' - w h' + (k'w + 1 / S) h h'
// and the adjoint after the update of step k-1 is A' lam~, A' Lam~ A (A over s_k - s_(k-1), identity on the b-block).
// Only scalar divisions (by S); no matrix is inverted.
template <int KID, int L>
__global__ void __launch_bounds__(32) ss_adjoint_kernel(SSProblem p, const double* __restrict__ hyp, const int* __restrict__ info,
                                                        SSStore st) {
    constexpr int d = ss::Dim<KID>::d, D = d + L, NP = D * (D + 1) / 2;
    if (threadIdx.x != 0 || *info != 0) return;
    double al[L];
    int cnt[L];
#pragma unroll
    for (int l = 0; l < L; ++l) { al[l] = hyp[L + l]; cnt[l] = p.band_start[l + 1]; }
    ss::Coef<d> c;
    ss::setup<KID>(hyp[2 * L], c);
    double lam[D], Lam[NP];
#pragma unroll
    for (int i = 0; i < D; ++i) lam[i] = 0.0;
#pragma unroll
    for (int i = 0; i < NP; ++i) Lam[i] = 0.0;
    for (int k = p.N - 1; k >= 0; --k) {
        const int l = st.band[k];
        int idx = 0;
        double a = 0.0;
#pragma unroll
        for (int lb = 0; lb < L; ++lb)
            if (lb == l) { idx = --cnt[lb]; a = al[lb]; }       // the k-th step of band l is its next sorted point, backwards
        const double r = p.r[idx], s2 = p.s2[idx];
        double m[D], P[NP];
        double A[d][d], Q[d][d], dA[d][d], dQ[d][d];
        const double Dt = k > 0 ? st.t[k] - st.t[k - 1] : 0.0;
        if (k > 0) {
#pragma unroll
            for (int i = 0; i < D; ++i) m[i] = st.m[(size_t)(k - 1) * D + i];
#pragma unroll
            for (int i = 0; i < NP; ++i) P[i] = st.P[(size_t)(k - 1) * NP + i];
        } else {
            prior_moments<KID, L>(c, p, m, P);
        }
        if (Dt > 0.0) {
            ss::step<KID, false>(c, Dt, A, Q, dA, dQ);
            ss::predict_moments<d, D>(A, Q, m, P);
        }
        double h[D], Ph[D];
#pragma unroll
        for (int i = 0; i < D; ++i) {
            h[i] = i == 0 ? a : (i >= d && i - d == l) ? 1.0 : 0.0;
            double s = 0.0;
#pragma unroll
            for (int lb = 0; lb < L; ++lb)
                if (lb == l) s = P[sym<D>(i, d + lb)];
            Ph[i] = fma(a, P[sym<D>(i, 0)], s);
        }
        double Phb = 0.0, mb = 0.0;
#pragma unroll
        for (int lb = 0; lb < L; ++lb)
            if (lb == l) { Phb = Ph[d + lb]; mb = m[d + lb]; }
        const double S = fma(a, Ph[0], Phb) + s2;            // the filter's innovation variance and residual
        const double v = r - fma(a, m[0], mb);
        const double iS = 1.0 / S;
        double kg[D], w[D], kl = 0.0, kw = 0.0;
#pragma unroll
        for (int i = 0; i < D; ++i) kg[i] = Ph[i] * iS;
#pragma unroll
        for (int i = 0; i < D; ++i) {
            double s = 0.0;
#pragma unroll
            for (int q = 0; q < D; ++q) s = fma(Lam[sym<D>(i, q)], kg[q], s);
            w[i] = s;
            kl = fma(kg[i], lam[i], kl);
        }
#pragma unroll
        for (int i = 0; i < D; ++i) kw = fma(kg[i], w[i], kw);
        const double cl = fma(v, iS, kl), cL = kw + iS;
#pragma unroll
        for (int i = 0; i < D; ++i) lam[i] = fma(-h[i], cl, lam[i]);
#pragma unroll
        for (int i = 0; i < D; ++i)
#pragma unroll
            for (int q = i; q < D; ++q)
                Lam[sym<D>(i, q)] = fma(cL * h[i], h[q], Lam[sym<D>(i, q)] - fma(h[i], w[q], w[i] * h[q]));
#pragma unroll
        for (int i = 0; i < D; ++i) st.lam[(size_t)k * D + i] = lam[i];
#pragma unroll
        for (int i = 0; i < NP; ++i) st.Lam[(size_t)k * NP + i] = Lam[i];
        if (k > 0 && Dt > 0.0) {
            double lf[d], B[d][d];
#pragma unroll
            for (int i = 0; i < d; ++i) {
                double s = 0.0;
#pragma unroll
                for (int q = 0; q < d; ++q) s = fma(A[q][i], lam[q], s);
                lf[i] = s;
            }
#pragma unroll
            for (int i = 0; i < d; ++i) lam[i] = lf[i];
#pragma unroll
            for (int kc = d; kc < D; ++kc) {            // Lam_fb = A' Lam_fb
#pragma unroll
                for (int i = 0; i < d; ++i) {
                    double s = 0.0;
#pragma unroll
                    for (int q = 0; q < d; ++q) s = fma(A[q][i], Lam[sym<D>(q, kc)], s);
                    lf[i] = s;
                }
#pragma unroll
                for (int i = 0; i < d; ++i) Lam[sym<D>(i, kc)] = lf[i];
            }
#pragma unroll
            for (int i = 0; i < d; ++i)                 // B = Lam_ff A, then Lam_ff = A' B
#pragma unroll
                for (int j = 0; j < d; ++j) {
                    double s = 0.0;
#pragma unroll
                    for (int q = 0; q < d; ++q) s = fma(Lam[sym<D>(i, q)], A[q][j], s);
                    B[i][j] = s;
                }
#pragma unroll
            for (int i = 0; i < d; ++i)
#pragma unroll
                for (int j = i; j < d; ++j) {
                    double s = 0.0;
#pragma unroll
                    for (int q = 0; q < d; ++q) s = fma(A[q][i], B[q][j], s);
                    Lam[sym<D>(i, j)] = s;
                }
        }
    }
}

// One thread per test point, in input order: the last stored step at or before its shifted time (binary search; a test
// time equal to a training time sits after it), then ss::point_moments.
template <int KID, int L>
__global__ void __launch_bounds__(128) ss_point_kernel(SSProblem p, const double* __restrict__ hyp, SSStore st, int NT,
                                                       const double* __restrict__ tt, const int* __restrict__ bt,
                                                       double* __restrict__ mu, double* __restrict__ sd) {
    constexpr int d = ss::Dim<KID>::d, D = d + L, NP = D * (D + 1) / 2;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= NT) return;
    const int l = bt[j];
    const double ts = tt[j] - hyp[l], a = hyp[L + l];
    ss::Coef<d> c;
    ss::setup<KID>(hyp[2 * L], c);
    int lo = 0, hi = p.N;                          // first step with s > ts
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (st.t[mid] <= ts) lo = mid + 1; else hi = mid;
    }
    const int i = lo - 1;
    double m[D], P[NP];
    if (i >= 0) {
#pragma unroll
        for (int q = 0; q < D; ++q) m[q] = st.m[(size_t)i * D + q];
#pragma unroll
        for (int q = 0; q < NP; ++q) P[q] = st.P[(size_t)i * NP + q];
    } else {
        prior_moments<KID, L>(c, p, m, P);          // stationary: no propagation to ts
    }
    const bool later = i + 1 < p.N;
    double mean, var;
    ss::point_moments<KID, L>(c, l, a, m, P, i >= 0 ? ts - st.t[i] : 0.0, later ? st.lam + (size_t)(i + 1) * D : nullptr,
                              later ? st.Lam + (size_t)(i + 1) * NP : nullptr, later ? st.t[i + 1] - ts : 0.0, mean, var);
    mu[j] = mean + p.mub[l];
    if (sd) sd[j] = sqrt(fmax(var + JITTER, SIGMA_FLOOR));
}

template <int KID, int L>
cudaError_t store_l(const SSProblem& p, const double* hyp, double* ll, int* info, const SSStore& st, cudaStream_t stream) {
    if (p.L == L) {
        ss_filter_kernel<KID, L, false, true><<<1, 32, 0, stream>>>(p, 1, hyp, hyp + L, hyp + 2 * L, ll, nullptr, info, nullptr, st);
        ss_adjoint_kernel<KID, L><<<1, 32, 0, stream>>>(p, hyp, info, st);
        return cudaGetLastError();
    }
    if constexpr (L < MAX_BANDS) return store_l<KID, L + 1>(p, hyp, ll, info, st, stream);
    return cudaErrorInvalidValue;
}

template <int KID, int L>
cudaError_t point_l(const SSProblem& p, const double* hyp, const SSStore& st, int NT, const double* tt, const int* bt,
                    double* mu, double* sd, cudaStream_t stream) {
    if (p.L == L) {
        ss_point_kernel<KID, L><<<(NT + 127) / 128, 128, 0, stream>>>(p, hyp, st, NT, tt, bt, mu, sd);
        return cudaGetLastError();
    }
    if constexpr (L < MAX_BANDS) return point_l<KID, L + 1>(p, hyp, st, NT, tt, bt, mu, sd, stream);
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

namespace gpcc {

cudaError_t statespace_store_launch(int kernel_id, const SSProblem& p, const double* hyp, double* ll, int* info,
                                    const SSStore& st, cudaStream_t stream) {
    switch (kernel_id) {
        case K_OU:  return store_l<K_OU, 1>(p, hyp, ll, info, st, stream);
        case K_M32: return store_l<K_M32, 1>(p, hyp, ll, info, st, stream);
        case K_M52: return store_l<K_M52, 1>(p, hyp, ll, info, st, stream);
        default:    return cudaErrorInvalidValue;
    }
}

cudaError_t statespace_predict_launch(int kernel_id, const SSProblem& p, const double* hyp, const SSStore& st, int NT,
                                      const double* tt, const int* bt, double* mu, double* sd, cudaStream_t stream) {
    if (NT <= 0) return cudaSuccess;
    switch (kernel_id) {
        case K_OU:  return point_l<K_OU, 1>(p, hyp, st, NT, tt, bt, mu, sd, stream);
        case K_M32: return point_l<K_M32, 1>(p, hyp, st, NT, tt, bt, mu, sd, stream);
        case K_M52: return point_l<K_M52, 1>(p, hyp, st, NT, tt, bt, mu, sd, stream);
        default:    return cudaErrorInvalidValue;
    }
}

}  // namespace gpcc
