// Exact O(N) joint posterior draws of the state-space fit state (gpcc_ss_state_sample): draws of
// g*_j = alpha_l f(t*_j - tau_l) + b_l + eta_j, eta_j ~ N(0, 1e-8), at test times of any band, distributed as N(mu_pred,
// Sigma_pred) of pred(::Vector{Vector}) (gpccfixdelay_marginaliseb.jl:259-289) without an N x N or NT x NT matrix.
//
// Pathwise conditioning (Matheron's rule), in the state's residual form r = y - mu_b, x = [f-state (d); b' (L)]:
//   1. a joint prior draw over the training and test times: f~ from the scan sampler of ss_sample.cu over the merged problem
//      (training points with their sigma_i^2, test points with sigma^2 = 1e-8, the jitter), b~'_l = sqrt(Sigma_b,l) zeta_l;
//      the data draw is y~'_i = f~_i + b~'_l and the test draw g~*_j = mu_b,l + b~'_l + f~_(N+j);
//   2. pseudo-residuals d_i = r_i - y~'_i;
//   3. the zero-mean smoother mean of d with the state's own gains: a forward mean pass m- = A m, v = d - h'm-, m = m- + k v,
//      and a backward pass of the mean part of the Bryson-Frazier adjoint, lam~ = lam^ - h (k'lam^ + v / S), lam^ <- A' lam~
//      (the recursion of ss_adjoint_kernel, statespace.cu, restricted to lam); at a test point the correction is the mean of
//      ss::point_moments, c1'm - w'lam~ (ss::point_mean_weights);
//   4. draw = g~* + correction.  The gains do not depend on the data, so its mean is mu_pred and its covariance Sigma_pred.
//
// Kernels:
//   - ss_ps_record_kernel (once per state): per merged training step, A over the gap before it, the gain k = P- h / S, 1 / S,
//     alpha_l and the residual, from the stored P of the step before with the filter's own predict (as ss_adjoint_kernel);
//   - ss_ps_locate_kernel (once per call): per test point, the last training step at or before it (the binary search of
//     ss_point_kernel) and its weights c1, w; it flags the steps whose m (bit 0) or lam~ (bit 1) a test point reads;
//   - per chunk of samples: ss_ps_shift_kernel (b~'), ss_ps_pseudo_kernel (d, layout [step][sample]), ss_ps_forward_kernel
//     and ss_ps_backward_kernel (one thread per sample, one sequential chain of N steps each; the threads of a warp walk the
//     same steps, so every record load is a broadcast), ss_ps_point_kernel (one thread per (test point, sample)).
// The passes keep v for every step and m, lam~ only at flagged steps, in slots numbered in pass order; the first thread of the
// first chunk writes the slot of every flagged step (mpos, lpos) for the point kernel.
#include "gpcc_internal.h"
#include "kernfun.cuh"
#include "philox.cuh"
#include "ss_model.h"

namespace gpcc {
namespace {

using ss::sym;

template <int KID, int L> struct PS {           // one record: A (d x d), k (D), 1 / S, alpha_l, residual
    static constexpr int d = ss::Dim<KID>::d, D = d + L, NP = D * (D + 1) / 2, W = d * d + D + 3;
    static constexpr int K = d * d, IS = K + D, AL = IS + 1, R = AL + 1;
};

template <int KID, int L>
__device__ __forceinline__ void prior_P(const ss::Coef<ss::Dim<KID>::d>& c, const double* Sigmab, double (&P)[PS<KID, L>::NP]) {
    constexpr int d = ss::Dim<KID>::d, D = d + L;
#pragma unroll
    for (int i = 0; i < D; ++i)
#pragma unroll
        for (int k = i; k < D; ++k) P[sym<D>(i, k)] = k < d ? c.Pinf[i][k] : i == k ? Sigmab[i - d] : 0.0;
}

// p: the training problem (each band sorted, on the device); order: merged step -> sorted point (ss_rank_kernel).
template <int KID, int L>
__global__ void __launch_bounds__(128) ss_ps_record_kernel(SSProblem p, const double* __restrict__ hyp, SSStore st,
                                                           const int* __restrict__ order, const int* __restrict__ perm,
                                                           double* __restrict__ rec, int* __restrict__ in) {
    using R = PS<KID, L>;
    constexpr int d = R::d, D = R::D, NP = R::NP;
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= p.N) return;
    const int j = order[k], l = st.band[k];
    const double a = hyp[L + l];
    ss::Coef<d> c;
    ss::setup<KID>(hyp[2 * L], c);
    double m[D], P[NP], A[d][d], Q[d][d], dA[d][d], dQ[d][d];
#pragma unroll
    for (int i = 0; i < D; ++i) m[i] = 0.0;
    if (k > 0) {
#pragma unroll
        for (int i = 0; i < NP; ++i) P[i] = st.P[(size_t)(k - 1) * NP + i];
    } else {
        prior_P<KID, L>(c, p.Sigmab, P);
    }
#pragma unroll
    for (int i = 0; i < d; ++i)
#pragma unroll
        for (int q = 0; q < d; ++q) A[i][q] = i == q ? 1.0 : 0.0;
    const double Dt = k > 0 ? st.t[k] - st.t[k - 1] : 0.0;
    if (Dt > 0.0) {
        ss::step<KID, false>(c, Dt, A, Q, dA, dQ);
        ss::predict_moments<d, D>(A, Q, m, P);
    }
    double Ph[D];
#pragma unroll
    for (int i = 0; i < D; ++i) {
        double s = 0.0;
#pragma unroll
        for (int lb = 0; lb < L; ++lb)
            if (lb == l) s = P[sym<D>(i, d + lb)];
        Ph[i] = fma(a, P[sym<D>(i, 0)], s);
    }
    double Phb = 0.0;
#pragma unroll
    for (int lb = 0; lb < L; ++lb)
        if (lb == l) Phb = Ph[d + lb];
    const double iS = 1.0 / (fma(a, Ph[0], Phb) + p.s2[j]);     // the filter's innovation variance
    double* r = rec + (size_t)k * R::W;
#pragma unroll
    for (int i = 0; i < d; ++i)
#pragma unroll
        for (int q = 0; q < d; ++q) r[i * d + q] = A[i][q];
#pragma unroll
    for (int i = 0; i < D; ++i) r[R::K + i] = Ph[i] * iS;
    r[R::IS] = iS;
    r[R::AL] = a;
    r[R::R] = p.r[j];
    in[k] = perm[j];
}

// One thread per test point: its step i (-1 before the first), the weights [c1 (D), w (D)], and the flags of steps i and i+1.
template <int KID, int L>
__global__ void __launch_bounds__(128) ss_ps_locate_kernel(SSProblem p, const double* __restrict__ hyp, SSStore st, int NT,
                                                           const double* __restrict__ tt, const int* __restrict__ bt,
                                                           int* __restrict__ tstep, double* __restrict__ tw, int* need) {
    using R = PS<KID, L>;
    constexpr int d = R::d, D = R::D, NP = R::NP;
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
    double P[NP];
    if (i >= 0) {
#pragma unroll
        for (int q = 0; q < NP; ++q) P[q] = st.P[(size_t)i * NP + q];
    } else {
        prior_P<KID, L>(c, p.Sigmab, P);
    }
    const bool later = i + 1 < p.N;
    double c1[D], w[D];
    ss::point_mean_weights<KID, L>(c, l, a, P, i >= 0 ? ts - st.t[i] : 0.0, later, later ? st.t[i + 1] - ts : 0.0, c1, w);
    tstep[j] = i;
#pragma unroll
    for (int q = 0; q < D; ++q) { tw[(size_t)j * 2 * D + q] = c1[q]; tw[(size_t)j * 2 * D + D + q] = w[q]; }
    if (i >= 0) atomicOr(need + i, 1);
    if (later) atomicOr(need + i + 1, 2);
}

// b~'[s][l] = sqrt(Sigma_b,l) zeta; zeta from the caller or from Philox counter (l, sample, tag, 2): the point deviates of
// ss_sample.cu use the last counter word 0 and 1 only.
__global__ void __launch_bounds__(128) ss_ps_shift_kernel(SSPostArgs a) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= a.C * a.L) return;
    const int s = g / a.L, l = g - s * a.L;
    double z;
    if (a.zin_b) {
        z = a.zin_b[g];
    } else {
        const uint2 key = make_uint2((unsigned)a.seed, (unsigned)(a.seed >> 32));
        z = box_muller(philox4x32_10(make_uint4((unsigned)l, (unsigned)(a.sample0 + s), a.tag, 2u), key)).x;
    }
    if (a.zout_b) a.zout_b[g] = z;
    a.bs[g] = a.sqrt_sigmab[l] * z;
}

// d[k][s] = r - f~ - b~' at training step k
template <int W>
__global__ void __launch_bounds__(256) ss_ps_pseudo_kernel(SSPostArgs a) {
    const size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= (size_t)a.N * a.C) return;
    const int k = (int)(g / (size_t)a.C), s = (int)(g - (size_t)k * a.C);
    a.dv[g] = a.rec[(size_t)k * W + W - 1] - a.f[(size_t)s * a.NM + a.in[k]] - a.bs[(size_t)s * a.L + a.band[k]];
}

template <int KID, int L>
__global__ void __launch_bounds__(128) ss_ps_forward_kernel(SSPostArgs a) {
    using R = PS<KID, L>;
    constexpr int d = R::d, D = R::D;
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= a.C) return;
    const bool first = a.sample0 == 0 && s == 0;
    const size_t C = (size_t)a.C;
    double m[D];
#pragma unroll
    for (int i = 0; i < D; ++i) m[i] = 0.0;
    int cnt = 0;
    for (int k = 0; k < a.N; ++k) {
        const double* __restrict__ r = a.rec + (size_t)k * R::W;
        const int l = __ldg(a.band + k);
        if (k > 0) {                               // m_f = A m_f (A = I on a tie)
            double mf[d];
#pragma unroll
            for (int i = 0; i < d; ++i) {
                double t = 0.0;
#pragma unroll
                for (int q = 0; q < d; ++q) t = fma(__ldg(r + i * d + q), m[q], t);
                mf[i] = t;
            }
#pragma unroll
            for (int i = 0; i < d; ++i) m[i] = mf[i];
        }
        double mb = 0.0;
#pragma unroll
        for (int lb = 0; lb < L; ++lb)
            if (lb == l) mb = m[d + lb];
        const double v = a.dv[k * C + s] - fma(__ldg(r + R::AL), m[0], mb);
#pragma unroll
        for (int i = 0; i < D; ++i) m[i] = fma(__ldg(r + R::K + i), v, m[i]);
        a.dv[k * C + s] = v;
        if (__ldg(a.need + k) & 1) {
#pragma unroll
            for (int q = 0; q < D; ++q) a.mbuf[((size_t)cnt * D + q) * C + s] = m[q];
            if (first) a.mpos[k] = cnt;
            ++cnt;
        }
    }
}

template <int KID, int L>
__global__ void __launch_bounds__(128) ss_ps_backward_kernel(SSPostArgs a) {
    using R = PS<KID, L>;
    constexpr int d = R::d, D = R::D;
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= a.C) return;
    const bool first = a.sample0 == 0 && s == 0;
    const size_t C = (size_t)a.C;
    double lam[D];
#pragma unroll
    for (int i = 0; i < D; ++i) lam[i] = 0.0;
    int cnt = 0;
    for (int k = a.N - 1; k >= 0; --k) {
        const double* __restrict__ r = a.rec + (size_t)k * R::W;
        const int l = __ldg(a.band + k);
        double kl = 0.0;
#pragma unroll
        for (int i = 0; i < D; ++i) kl = fma(__ldg(r + R::K + i), lam[i], kl);
        const double cl = fma(a.dv[k * C + s], __ldg(r + R::IS), kl);
        lam[0] = fma(-__ldg(r + R::AL), cl, lam[0]);          // lam~ = lam^ - h cl, h = alpha_l e_0 + e_(d+l)
#pragma unroll
        for (int lb = 0; lb < L; ++lb)
            if (lb == l) lam[d + lb] -= cl;
        if (__ldg(a.need + k) & 2) {
#pragma unroll
            for (int q = 0; q < D; ++q) a.lbuf[((size_t)cnt * D + q) * C + s] = lam[q];
            if (first) a.lpos[k] = cnt;
            ++cnt;
        }
        if (k > 0) {                               // lam_f = A' lam_f
            double lf[d];
#pragma unroll
            for (int i = 0; i < d; ++i) {
                double t = 0.0;
#pragma unroll
                for (int q = 0; q < d; ++q) t = fma(__ldg(r + q * d + i), lam[q], t);
                lf[i] = t;
            }
#pragma unroll
            for (int i = 0; i < d; ++i) lam[i] = lf[i];
        }
    }
}

// out[s][j] = mu_b,l + b~'_l + f~_(N+j) + c1'm_i - w'lam~_(i+1)
template <int D>
__global__ void __launch_bounds__(128) ss_ps_point_kernel(SSPostArgs a) {
    const size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= (size_t)a.NT * a.C) return;
    const size_t C = (size_t)a.C;
    const int j = (int)(g / C), s = (int)(g - (size_t)j * C);
    const int i = a.tstep[j], l = a.bt[j];
    const double* w = a.tw + (size_t)j * 2 * D;
    double corr = 0.0;
    if (i >= 0) {
        const double* m = a.mbuf + (size_t)a.mpos[i] * D * C + s;
#pragma unroll
        for (int q = 0; q < D; ++q) corr = fma(w[q], m[q * C], corr);
    }
    if (i + 1 < a.N) {
        const double* lam = a.lbuf + (size_t)a.lpos[i + 1] * D * C + s;
#pragma unroll
        for (int q = 0; q < D; ++q) corr = fma(-w[D + q], lam[q * C], corr);
    }
    a.out[(size_t)s * a.NT + j] = (a.mub[l] + a.bs[(size_t)s * a.L + l]) + a.f[(size_t)s * a.NM + a.N + j] + corr;
}

template <int KID, int L>
cudaError_t records_l(const SSProblem& p, const double* hyp, const SSStore& st, const int* order, const int* perm,
                      double* rec, int* in, cudaStream_t stream) {
    if (p.L == L) {
        ss_ps_record_kernel<KID, L><<<(p.N + 127) / 128, 128, 0, stream>>>(p, hyp, st, order, perm, rec, in);
        return cudaGetLastError();
    }
    if constexpr (L < MAX_BANDS) return records_l<KID, L + 1>(p, hyp, st, order, perm, rec, in, stream);
    return cudaErrorInvalidValue;
}

template <int KID, int L>
cudaError_t locate_l(const SSProblem& p, const double* hyp, const SSStore& st, int NT, const double* tt, const int* bt,
                     int* tstep, double* tw, int* need, cudaStream_t stream) {
    if (p.L == L) {
        ss_ps_locate_kernel<KID, L><<<(NT + 127) / 128, 128, 0, stream>>>(p, hyp, st, NT, tt, bt, tstep, tw, need);
        return cudaGetLastError();
    }
    if constexpr (L < MAX_BANDS) return locate_l<KID, L + 1>(p, hyp, st, NT, tt, bt, tstep, tw, need, stream);
    return cudaErrorInvalidValue;
}

template <int KID, int L>
cudaError_t chunk_l(const SSPostArgs& a, cudaStream_t stream) {
    if (a.L == L) {
        using R = PS<KID, L>;
        const size_t nd = (size_t)a.N * a.C, np = (size_t)a.NT * a.C;
        if ((nd + 255) / 256 > 0x7fffffffu || (np + 127) / 128 > 0x7fffffffu) return cudaErrorInvalidValue;
        const unsigned bs = (unsigned)((a.C + 127) / 128);
        ss_ps_shift_kernel<<<(a.C * a.L + 127) / 128, 128, 0, stream>>>(a);
        ss_ps_pseudo_kernel<R::W><<<(unsigned)((nd + 255) / 256), 256, 0, stream>>>(a);
        ss_ps_forward_kernel<KID, L><<<bs, 128, 0, stream>>>(a);
        ss_ps_backward_kernel<KID, L><<<bs, 128, 0, stream>>>(a);
        ss_ps_point_kernel<R::D><<<(unsigned)((np + 127) / 128), 128, 0, stream>>>(a);
        return cudaGetLastError();
    }
    if constexpr (L < MAX_BANDS) return chunk_l<KID, L + 1>(a, stream);
    return cudaErrorInvalidValue;
}

}  // namespace

int statespace_post_record_width(int kernel_id, int L) {
    const int d = kernel_id == K_OU ? 1 : kernel_id == K_M32 ? 2 : 3;
    return d * d + d + L + 3;
}

cudaError_t statespace_post_records_launch(int kernel_id, const SSProblem& p, const double* hyp, const double* h_tau,
                                           const SSStore& st, const int* perm, int* order, double* rec, int* in,
                                           cudaStream_t stream) {
    cudaError_t e = statespace_rank_launch(p, h_tau, order, stream);
    if (e != cudaSuccess) return e;
    switch (kernel_id) {
        case K_OU:  return records_l<K_OU, 1>(p, hyp, st, order, perm, rec, in, stream);
        case K_M32: return records_l<K_M32, 1>(p, hyp, st, order, perm, rec, in, stream);
        case K_M52: return records_l<K_M52, 1>(p, hyp, st, order, perm, rec, in, stream);
        default:    return cudaErrorInvalidValue;
    }
}

cudaError_t statespace_post_locate_launch(int kernel_id, const SSProblem& p, const double* hyp, const SSStore& st, int NT,
                                          const double* tt, const int* bt, int* tstep, double* tw, int* need,
                                          cudaStream_t stream) {
    if (NT <= 0) return cudaSuccess;
    switch (kernel_id) {
        case K_OU:  return locate_l<K_OU, 1>(p, hyp, st, NT, tt, bt, tstep, tw, need, stream);
        case K_M32: return locate_l<K_M32, 1>(p, hyp, st, NT, tt, bt, tstep, tw, need, stream);
        case K_M52: return locate_l<K_M52, 1>(p, hyp, st, NT, tt, bt, tstep, tw, need, stream);
        default:    return cudaErrorInvalidValue;
    }
}

cudaError_t statespace_post_chunk_launch(int kernel_id, const SSPostArgs& a, cudaStream_t stream) {
    if (a.N <= 0 || a.NT <= 0 || a.C <= 0) return cudaErrorInvalidValue;
    switch (kernel_id) {
        case K_OU:  return chunk_l<K_OU, 1>(a, stream);
        case K_M32: return chunk_l<K_M32, 1>(a, stream);
        case K_M52: return chunk_l<K_M52, 1>(a, stream);
        default:    return cudaErrorInvalidValue;
    }
}

}  // namespace gpcc
