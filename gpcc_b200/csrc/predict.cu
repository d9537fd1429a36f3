// The fitted state behind `postb` and the `pred` closures (SURVEY.md rows a9, a10, f1; K5, K6).
//   gpcc_fit_state_create          src/gpccfixdelay_marginaliseb.jl:235-252  (what the reference's closures capture: KSobsB, postb)
//   gpcc_fit_state_postb           :248-252
//   gpcc_fit_state_predict         :259-307
//   gpcc_fit_state_predict_loglik  :311-343
//   gpcc_postb / gpcc_predict / gpcc_predict_loglik: the same through a one-entry cache on the problem.
//
// The reference factorises KSobsB = K + Sobs + B with a dense `\` (LU) on EVERY pred call (:275, :283) and K + Sobs twice
// more for postb (:248-250).  Here ONE Cholesky factorisation per fitted (delays, alpha, rho) is kept on the device:
// A = K + Sobs = Lc Lc' (the tiled DMMA path of large_path.cu in forward mode, any N), together with
//     V = Lc^-1 Q,  u = Lc^-1 Y,  Sigma_postb = (Sigma_b^-1 + V'V)^-1,  mu_postb = Sigma_postb (V'u + Sigma_b^-1 mu_b)   (= :248-250)
//     w = u - V mu_postb = Lc^-1 (Y - Q mu_postb).
// A prediction is then a rectangular assembly k* (WITHOUT the B term), one triangular solve Z = Lc^-1 k* and reductions:
//     mu_pred    = Z'w + Q* mu_postb
//     Sigma_pred = c** - Z'Z + R' Sigma_postb R + 1e-8 I,    R = Q*' - V'Z.
// This is the reference's  kB*'(KSobsB \ (Y - bbar)) + Q* mu_b  and  cB - kB*'(KSobsB \ kB*)  (:275-285) with the rank-L term
// B = Q Sigma_b Q' carried through the Woodbury identity instead of inside the matrix (Rasmussen & Williams 2006, eq. 2.41-2.42
// with a Gaussian prior on the explicit basis coefficients).  Reason: Sigma_b = 100 var(y) ~ 1e3 while sigma_pred^2 ~ 0.1, so the
// reference's form subtracts two numbers of size Sigma_b and loses ~4 digits on top of cond(K) eps; the form above never forms
// a quantity of size Sigma_b and is held to 1e-8 against 50-digit arithmetic (tests/golden/pred_exact.npz).
#include "state.h"
#include "kernfun.cuh"
#include <cmath>
#include <cstring>
#include <limits>

using namespace gpcc;

namespace {

constexpr double JITTER = 1e-8;       // :69, :279
constexpr double SIGMA_FLOOR = 1e-6;  // :303
constexpr double LOG2PI = 1.8378770664093454835606594728112;

struct HyperDev {   // small by-value parameter block
    double delays[GPCC_MAX_BANDS];
    double alpha[GPCC_MAX_BANDS];
    double rho;
    int L;
};

struct PostB {      // posterior of the shifts, device resident
    double mu[GPCC_MAX_BANDS];
    double S[GPCC_MAX_BANDS][GPCC_MAX_BANDS];
};

template <class T>
struct GrowBuf {    // device buffer that only ever grows (no cudaMalloc on repeated calls of the same size)
    T* d = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (d) cudaFree(d);
        d = nullptr; cap = 0;
        cudaError_t e = cudaMalloc(&d, std::max<size_t>(n, 1) * sizeof(T));
        if (e == cudaSuccess) cap = n;
        return e;
    }
    void release() { if (d) cudaFree(d); d = nullptr; cap = 0; }
};

}  // namespace

struct gpcc_fit_state {
    gpcc_problem* p = nullptr;
    int dev = 0;
    int N = 0, L = 0, kernel_id = 0;
    HyperDev h{};
    double* Lc = nullptr;      // [N][N] column-major Cholesky factor of K + Sobs (lower)
    double* VU = nullptr;      // [N][L+1] column-major: V = Lc^-1 Q, last column u = Lc^-1 Y
    double* w = nullptr;       // [N]  Lc^-1 (Y - Q mu_postb)
    PostB* postb_d = nullptr;  // device copy
    PostB postb_h{};           // host copy
    int* band_start_d = nullptr;
    // scratch of the prediction calls, kept between calls
    GrowBuf<double> Z, R, G, S, mu, sd, tt, extra, yv, zv, scal;
    GrowBuf<int> bandt, info;
    long long n_factorisations = 0;   // diagnostics: how often the N^3 work ran for this state (must stay 1)
};

namespace {

// ---------------------------------------------------------------------------------------------------------------------
// k* = delayedCovariance(kernel, alpha, tau, rho, tarray, ttest)  (:269 without the B* term), column-major N x NT
// ---------------------------------------------------------------------------------------------------------------------
template <int KID>
__global__ void cross_cov_kernel(int N, int NT, const double* __restrict__ t, const int* __restrict__ band,
                                 const double* __restrict__ tt, const int* __restrict__ bandt, HyperDev h,
                                 double* __restrict__ out) {
    const KernParams kp = make_kern_params(KID, h.rho);
    for (int j = blockIdx.y; j < NT; j += gridDim.y) {
        const int bj = bandt[j];
        const double tj = tt[j] - h.delays[bj], aj = h.alpha[bj];
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) {
            const int bi = band[i];
            out[(size_t)j * N + i] = (h.alpha[bi] * aj) * kern_value<KID>((t[i] - h.delays[bi]) - tj, kp);   // delayedCovariance.jl:27
        }
    }
}

// [Q | Y]: the right-hand sides of the state (util.jl:56-70 Qmatrix; :85 Y), column-major N x (L+1)
__global__ void rhs_qy_kernel(int N, int L, const int* __restrict__ band, const double* __restrict__ y, double* __restrict__ out) {
    for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < N * (L + 1); q += gridDim.x * blockDim.x) {
        const int i = q % N, c = q / N;
        out[q] = c < L ? (band[i] == c ? 1.0 : 0.0) : y[i];
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// X <- Lc^-1 X for a dense column-major lower-triangular Lc (N x N) and m right-hand sides (N x m, column-major).
// One CTA owns TC columns and walks down the matrix in blocks of TB rows: forward substitution inside the diagonal block
// (one warp per column, the column block in registers, pivot value broadcast with a shuffle), then a rank-TB update of all
// rows below (thread = row, coalesced reads of Lc, the solved block broadcast from shared memory).  FP64 FMA throughout;
// this is the backward-stable triangular solve that keeps sigma_pred at Cholesky accuracy.
// ---------------------------------------------------------------------------------------------------------------------
constexpr int TB = 64, TC = 8;
__global__ void __launch_bounds__(256) trsm_lower_kernel(int N, int m, const double* __restrict__ Lc, double* __restrict__ X) {
    __shared__ double Ld[TB][TB + 1];
    __shared__ double Xk[TB][TC];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int c0 = blockIdx.x * TC; c0 < m; c0 += gridDim.x * TC) {
        const int nc = min(TC, m - c0);
        for (int k0 = 0; k0 < N; k0 += TB) {
            const int nb = min(TB, N - k0);
            __syncthreads();
            for (int e = tid; e < TB * TB; e += 256) {
                const int r = e % TB, c = e / TB;
                Ld[r][c] = (r < nb && c <= r) ? Lc[(size_t)(k0 + c) * N + k0 + r] : (r == c ? 1.0 : 0.0);
            }
            __syncthreads();
            if (warp < nc) {
                double* col = X + (size_t)(c0 + warp) * N + k0;
                double x0 = lane < nb ? col[lane] : 0.0, x1 = lane + 32 < nb ? col[lane + 32] : 0.0;
                for (int j = 0; j < nb; ++j) {
                    const double mine = (j < 32 ? x0 : x1) / Ld[j][j];
                    const double xj = __shfl_sync(0xffffffffu, mine, j & 31);
                    if (lane == (j & 31)) { if (j < 32) x0 = xj; else x1 = xj; }
                    if (lane > j) x0 = fma(-Ld[lane][j], xj, x0);
                    if (lane + 32 > j) x1 = fma(-Ld[lane + 32][j], xj, x1);
                }
                if (lane < nb) col[lane] = x0;
                if (lane + 32 < nb) col[lane + 32] = x1;
                Xk[lane][warp] = x0;
                Xk[lane + 32][warp] = x1;
            } else if (warp < TC) {
                Xk[lane][warp] = 0.0;
                Xk[lane + 32][warp] = 0.0;
            }
            __syncthreads();
            for (int r = k0 + nb + tid; r < N; r += 256) {
                double acc[TC];
#pragma unroll
                for (int c = 0; c < TC; ++c) acc[c] = 0.0;
                for (int j = 0; j < nb; ++j) {
                    const double l = Lc[(size_t)(k0 + j) * N + r];
#pragma unroll
                    for (int c = 0; c < TC; ++c) acc[c] = fma(l, Xk[j][c], acc[c]);
                }
                for (int c = 0; c < nc; ++c) X[(size_t)(c0 + c) * N + r] -= acc[c];
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// State: G = V'V, hv = V'u, the L x L algebra of :248-252, then w = u - V mu_postb.  One CTA, deterministic reductions.
// ---------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) state_finish_kernel(int N, int L, const double* __restrict__ VU, const double* __restrict__ sigb,
                                                           const double* __restrict__ mub, PostB* __restrict__ out, double* __restrict__ w) {
    __shared__ double G[GPCC_MAX_BANDS][GPCC_MAX_BANDS + 1];
    __shared__ double red[8];
    __shared__ PostB pb;
    const int tid = threadIdx.x;
    for (int l = 0; l < L; ++l)
        for (int m = l; m <= L; ++m) {      // m == L: V'u
            double s = 0.0;
            for (int i = tid; i < N; i += 256) s = fma(VU[(size_t)l * N + i], VU[(size_t)m * N + i], s);
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            __syncthreads();
            if ((tid & 31) == 0) red[tid >> 5] = s;
            __syncthreads();
            if (tid == 0) {
                double v = 0.0;
                for (int q = 0; q < 8; ++q) v += red[q];
                G[l][m] = v;
                if (m < L) G[m][l] = v;
            }
        }
    __syncthreads();
    if (tid == 0) {
        // A = Sigma_b^-1 + Q'(Sobs+K)^-1 Q ; Sigma_post = A^-1 (Gauss-Jordan, A is SPD) (:248)
        double A[GPCC_MAX_BANDS][2 * GPCC_MAX_BANDS];
        for (int l = 0; l < L; ++l)
            for (int m = 0; m < L; ++m) {
                A[l][m] = G[l][m] + (l == m ? 1.0 / sigb[l] : 0.0);
                A[l][L + m] = (l == m) ? 1.0 : 0.0;
            }
        for (int k = 0; k < L; ++k) {
            const double pv = 1.0 / A[k][k];
            for (int m = 0; m < 2 * L; ++m) A[k][m] *= pv;
            for (int l = 0; l < L; ++l)
                if (l != k) {
                    const double f = A[l][k];
                    for (int m = 0; m < 2 * L; ++m) A[l][m] -= f * A[k][m];
                }
        }
        // mu_post = Sigma_post ((Q'/(Sobs+K)) Y + Sigma_b \ mu_b) (:250); Sigma_post symmetrised (:252)
        for (int l = 0; l < L; ++l) {
            double s = 0.0;
            for (int m = 0; m < L; ++m) s += A[l][L + m] * (G[m][L] + mub[m] / sigb[m]);
            pb.mu[l] = s;
            for (int m = 0; m < L; ++m) pb.S[l][m] = 0.5 * (A[l][L + m] + A[m][L + l]);
        }
        *out = pb;
    }
    __syncthreads();
    for (int i = tid; i < N; i += 256) {
        double s = VU[(size_t)L * N + i];
        for (int l = 0; l < L; ++l) s = fma(-VU[(size_t)l * N + i], pb.mu[l], s);
        w[i] = s;
    }
}

// One warp per test point j:  mu_j = Z_j'w + mu_postb[band*(j)] (:283-285);  R_lj = [l == band*(j)] - V_l'Z_j;
// var_j = alpha^2 k(0) - Z_j'Z_j + R_j' Sigma_postb R_j + JITTER (:272-279);  sd_j = sqrt(max(var_j, 1e-6)) (:303)
__global__ void col_stats_kernel(int N, int NT, int L, const double* __restrict__ Z, const double* __restrict__ VU,
                                 const double* __restrict__ w, const int* __restrict__ bandt, HyperDev h,
                                 const PostB* __restrict__ pbp, double* __restrict__ mu, double* __restrict__ R,
                                 double* __restrict__ sd) {
    const int j = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (j >= NT) return;
    const int lane = threadIdx.x & 31;
    double sm = 0.0, sq = 0.0, sv[GPCC_MAX_BANDS];
#pragma unroll
    for (int l = 0; l < GPCC_MAX_BANDS; ++l) sv[l] = 0.0;
    for (int i = lane; i < N; i += 32) {
        const double z = Z[(size_t)j * N + i];
        sm = fma(z, w[i], sm);
        sq = fma(z, z, sq);
#pragma unroll
        for (int l = 0; l < GPCC_MAX_BANDS; ++l)
            if (l < L) sv[l] = fma(z, VU[(size_t)l * N + i], sv[l]);
    }
    for (int o = 16; o > 0; o >>= 1) {
        sm += __shfl_xor_sync(0xffffffffu, sm, o);
        sq += __shfl_xor_sync(0xffffffffu, sq, o);
#pragma unroll
        for (int l = 0; l < GPCC_MAX_BANDS; ++l) sv[l] += __shfl_xor_sync(0xffffffffu, sv[l], o);
    }
    if (lane == 0) {
        const int b = bandt[j];
        double r[GPCC_MAX_BANDS];
#pragma unroll
        for (int l = 0; l < GPCC_MAX_BANDS; ++l) {
            r[l] = (l < L) ? ((l == b ? 1.0 : 0.0) - sv[l]) : 0.0;
            if (l < L) R[(size_t)j * L + l] = r[l];
        }
        double quad = 0.0;
        for (int l = 0; l < L; ++l)
            for (int m = 0; m < L; ++m) quad = fma(r[l] * pbp->S[l][m], r[m], quad);
        mu[j] = sm + pbp->mu[b];
        if (sd) sd[j] = sqrt(fmax(h.alpha[b] * h.alpha[b] - sq + quad + JITTER, SIGMA_FLOOR));
    }
}

// C[M x Nc] = A' B with A (K x M, lda = K) and B (K x Nc), column-major: the Gram matrix Z'Z.
__global__ void __launch_bounds__(256) gemm_tn_kernel(int M, int Nc, int K, const double* __restrict__ A,
                                                      const double* __restrict__ B, double* __restrict__ C) {
    __shared__ double As[16][65];
    __shared__ double Bs[16][65];
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int m0 = blockIdx.x * 64, n0 = blockIdx.y * 64;
    double acc[4][4] = {};
    for (int k0 = 0; k0 < K; k0 += 16) {
        for (int e = threadIdx.x; e < 16 * 64; e += 256) {
            const int kk = e & 15, mm = e >> 4;
            const int gm = m0 + mm, gn = n0 + mm, gk = k0 + kk;
            As[kk][mm] = (gm < M && gk < K) ? A[(size_t)gm * K + gk] : 0.0;
            Bs[kk][mm] = (gn < Nc && gk < K) ? B[(size_t)gn * K + gk] : 0.0;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < 16; ++kk) {
            double a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) { a[i] = As[kk][tx + 16 * i]; b[i] = Bs[kk][ty + 16 * i]; }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fma(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int gm = m0 + tx + 16 * i, gn = n0 + ty + 16 * j;
            if (gm < M && gn < Nc) C[(size_t)gn * M + gm] = acc[i][j];
        }
}

// Sigma_pred = c** - sym(Z'Z) + sym(R' Sigma_postb R) + JITTER I (:272-279), column-major NT x NT, bitwise symmetric;
// optional + diag(extra) (Sobs* of the test likelihood, :319)
template <int KID>
__global__ void pred_cov_kernel(int NT, int L, const double* __restrict__ G, const double* __restrict__ R,
                                const double* __restrict__ tt, const int* __restrict__ bandt, HyperDev h,
                                const PostB* __restrict__ pbp, const double* __restrict__ extra_diag, double* __restrict__ S) {
    const KernParams kp = make_kern_params(KID, h.rho);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= NT) return;
    for (int j = blockIdx.y; j < NT; j += gridDim.y) {
        const int bi = bandt[i], bj = bandt[j];
        const double d = fabs((tt[i] - h.delays[bi]) - (tt[j] - h.delays[bj]));      // |x - y|: the same bits for (i,j) and (j,i)
        const double c = (h.alpha[bi] * h.alpha[bj]) * kern_value<KID>(d, kp);
        double qij = 0.0, qji = 0.0;
        for (int l = 0; l < L; ++l)
            for (int m = 0; m < L; ++m) {
                qij = fma(R[(size_t)i * L + l] * pbp->S[l][m], R[(size_t)j * L + m], qij);
                qji = fma(R[(size_t)j * L + l] * pbp->S[l][m], R[(size_t)i * L + m], qji);
            }
        double v = c - 0.5 * (G[(size_t)j * NT + i] + G[(size_t)i * NT + j]) + 0.5 * (qij + qji);
        if (i == j) { v += JITTER; if (extra_diag) v += extra_diag[i]; }
        S[(size_t)j * NT + i] = v;
    }
}

// One-CTA right-looking Cholesky of an n x n column-major matrix in global memory followed by the Gaussian
// log-density of y under N(mu, S): out[0] = logpdf, info = k>0 if leading minor k is not PD.  (:325)
__global__ void __launch_bounds__(1024) chol_logpdf_kernel(int n, double* __restrict__ S, const double* __restrict__ y,
                                                           const double* __restrict__ mu, double* __restrict__ z,
                                                           double* __restrict__ out, int* __restrict__ info) {
    __shared__ double s_piv;
    __shared__ int s_info;
    __shared__ double red[32];
    const int tid = threadIdx.x, nt = blockDim.x;
    if (tid == 0) s_info = 0;
    for (int i = tid; i < n; i += nt) z[i] = y[i] - mu[i];
    __syncthreads();
    double logdet = 0.0;
    for (int k = 0; k < n; ++k) {
        if (tid == 0) {
            const double d = S[(size_t)k * n + k];
            if (!(d > 0.0) && s_info == 0) s_info = k + 1;
            s_piv = sqrt(d);
        }
        __syncthreads();
        if (s_info) break;
        const double piv = s_piv;
        for (int i = k + tid; i < n; i += nt) S[(size_t)k * n + i] /= piv;
        __syncthreads();
        // trailing update, lower triangle: column j (k<j<n), rows i>=j
        const int m = n - k - 1;
        for (long long e = tid; e < (long long)m * m; e += nt) {
            const int jj = (int)(e / m), ii = (int)(e % m);
            if (ii >= jj) {
                const int i = k + 1 + ii, j = k + 1 + jj;
                S[(size_t)j * n + i] -= S[(size_t)k * n + i] * S[(size_t)k * n + j];
            }
        }
        // forward substitution for z interleaved: z_k final, z_i -= L_ik z_k
        if (tid == 0) z[k] /= piv;
        __syncthreads();
        const double zk = z[k];
        for (int i = k + 1 + tid; i < n; i += nt) z[i] -= S[(size_t)k * n + i] * zk;
        logdet += 2.0 * log(piv);
        __syncthreads();
    }
    __syncthreads();
    if (s_info) { if (tid == 0) { *info = s_info; out[0] = -INFINITY; } return; }
    double q = 0.0;
    for (int i = tid; i < n; i += nt) q += z[i] * z[i];
    for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
    if ((tid & 31) == 0) red[tid >> 5] = q;
    __syncthreads();
    if (tid == 0) {
        double s = 0.0;
        for (int w = 0; w < (nt >> 5); ++w) s += red[w];
        out[0] = -0.5 * ((double)n * LOG2PI + logdet + s);
        *info = 0;
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// Sampling from the fitted process (the draw of src/simulatedata.jl:128-145, Y ~ MvNormal(0, C), on the device).
// Counter-based generator: Philox-4x32-10 (Salmon et al. 2011), counter = (index, 0, sample stream, 0), key = seed; two
// 53-bit uniforms per call -> Box-Muller pair.  Reproducible for a given seed whatever the launch geometry.
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const unsigned hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const unsigned hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u;
        k.y += 0xBB67AE85u;
    }
    return c;
}

__global__ void normal_kernel(size_t n, unsigned long long seed, double* __restrict__ z) {
    const uint2 key = make_uint2((unsigned)seed, (unsigned)(seed >> 32));
    for (size_t pair = (size_t)blockIdx.x * blockDim.x + threadIdx.x; 2 * pair < n; pair += (size_t)gridDim.x * blockDim.x) {
        const uint4 r = philox4x32_10(make_uint4((unsigned)pair, (unsigned)(pair >> 32), 0x47504343u, 0u), key);
        const double u1 = ((double)(((unsigned long long)(r.x >> 5) << 26) | (r.y >> 6)) + 0.5) * (1.0 / 9007199254740992.0);
        const double u2 = ((double)(((unsigned long long)(r.z >> 5) << 26) | (r.w >> 6)) + 0.5) * (1.0 / 9007199254740992.0);
        const double rad = sqrt(-2.0 * log(u1));
        double sn, cs;
        sincospi(2.0 * u2, &sn, &cs);
        z[2 * pair] = rad * cs;
        if (2 * pair + 1 < n) z[2 * pair + 1] = rad * sn;
    }
}

// f[s][i] = sum_{j <= i} Lc(i, j) z[s][j]: one thread per row, the rows of the column-major factor coalesced across threads
__global__ void __launch_bounds__(256) trmv_lower_kernel(int N, int ns, const double* __restrict__ Lc, const double* __restrict__ z,
                                                         double* __restrict__ f) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    for (int s0 = blockIdx.y * 4; s0 < ns; s0 += gridDim.y * 4) {
        double acc[4] = {0.0, 0.0, 0.0, 0.0};
        for (int j = 0; j <= i; ++j) {
            const double l = Lc[(size_t)j * N + i];
#pragma unroll
            for (int q = 0; q < 4; ++q)
                if (s0 + q < ns) acc[q] = fma(l, z[(size_t)(s0 + q) * N + j], acc[q]);
        }
#pragma unroll
        for (int q = 0; q < 4; ++q)
            if (s0 + q < ns) f[(size_t)(s0 + q) * N + i] = acc[q];
    }
}

int check_hyper(const gpcc_problem* p, const double* delays, const double* alpha, double rho) {
    if (!p || !delays || !alpha) return fail(-1, "NULL argument");
    for (int l = 0; l < p->L; ++l) {
        if (!(alpha[l] > 0) || !std::isfinite(alpha[l])) return fail(-2, "all(scale .> 0) violated (delayedCovariance.jl:3)");
        if (!std::isfinite(delays[l])) return fail(-3, "non-finite delay");
    }
    if (!(rho > 0) || !std::isfinite(rho)) return fail(-4, "rho is <= 0 (delayedCovariance.jl:5-7)");
    return 0;
}

void free_state(gpcc_fit_state* s) {
    cudaSetDevice(s->dev);
    for (void* q : {(void*)s->Lc, (void*)s->VU, (void*)s->w, (void*)s->postb_d, (void*)s->band_start_d}) if (q) cudaFree(q);
    s->Z.release(); s->R.release(); s->G.release(); s->S.release(); s->mu.release(); s->sd.release(); s->tt.release();
    s->extra.release(); s->yv.release(); s->zv.release(); s->scal.release(); s->bandt.release(); s->info.release();
    delete s;
}

int create_state(gpcc_problem* p, const double* delays, const double* alpha, double rho, gpcc_fit_state** out) {
    const int L = p->L, N = p->N;
    DeviceState& ds = p->ctx->ds[0];
    CUDA_TRY(cudaSetDevice(ds.dev));
    gpcc_fit_state* s = new gpcc_fit_state();
    s->p = p; s->dev = ds.dev; s->N = N; s->L = L; s->kernel_id = p->kernel_id;
    s->h.L = L; s->h.rho = rho;
    for (int l = 0; l < L; ++l) { s->h.delays[l] = delays[l]; s->h.alpha[l] = alpha[l]; }
    struct Guard { gpcc_fit_state* s; ~Guard() { if (s) free_state(s); } } guard{s};
    CUDA_TRY(cudaMalloc(&s->Lc, (size_t)N * N * sizeof(double)));
    CUDA_TRY(cudaMalloc(&s->VU, (size_t)N * (L + 1) * sizeof(double)));
    CUDA_TRY(cudaMalloc(&s->w, (size_t)N * sizeof(double)));
    CUDA_TRY(cudaMalloc(&s->postb_d, sizeof(PostB)));
    // ---- A = K + Sobs (no B) = Lc Lc': blocked right-looking Cholesky with DMMA trailing updates (large_path.cu) ----
    int rc = reserve_eval(p, 0, 1);
    if (rc) return rc;
    EvalSlot& q = ds.slot;
    std::memcpy(q.delays.h, delays, L * sizeof(double));
    std::memcpy(q.alpha.h, alpha, L * sizeof(double));
    q.rho.h[0] = rho;
    cudaStream_t st = ds.stream;
    CUDA_TRY(cudaMemcpyAsync(q.delays.d, q.delays.h, L * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(q.alpha.d, q.alpha.h, L * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(q.rho.d, q.rho.h, sizeof(double), cudaMemcpyHostToDevice, st));
    EvalBatch b;
    b.M = 1; b.delays = q.delays.d; b.alpha = q.alpha.d; b.rho = q.rho.d; b.want_grad = 0;
    b.ll = q.ll.d; b.grad = q.grad.d; b.info = q.info.d; b.mode_postb = 1; b.dump_chol = s->Lc;
    LargeTimings lt;
    CUDA_TRY(large_eval(p->pd[0].dp, b, ds.large, st, false, &lt));
    s->n_factorisations += 1;
    CUDA_TRY(cudaMemcpyAsync(q.info.h, q.info.d, sizeof(int), cudaMemcpyDeviceToHost, st));
    // ---- V = Lc^-1 Q, u = Lc^-1 Y, postb, w ----------------------------------------------------------------------
    const auto& dp = p->pd[0].dp;
    rhs_qy_kernel<<<(N * (L + 1) + 255) / 256, 256, 0, st>>>(N, L, dp.band, dp.y, s->VU);
    trsm_lower_kernel<<<(L + 1 + TC - 1) / TC, 256, 0, st>>>(N, L + 1, s->Lc, s->VU);
    CUDA_TRY(s->scal.reserve(2 * GPCC_MAX_BANDS + 2));
    CUDA_TRY(cudaMemcpyAsync(s->scal.d, p->Sigmab.data(), L * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(s->scal.d + GPCC_MAX_BANDS, p->mub.data(), L * sizeof(double), cudaMemcpyHostToDevice, st));
    state_finish_kernel<<<1, 256, 0, st>>>(N, L, s->VU, s->scal.d, s->scal.d + GPCC_MAX_BANDS, s->postb_d, s->w);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(&s->postb_h, s->postb_d, sizeof(PostB), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (q.info.h[0] != 0) return fail(-6, "K + Sobs is not positive definite for these hyper-parameters");
    ds.launches += lt.launches + 3;
    guard.s = nullptr;
    *out = s;
    return 0;
}

template <int KID>
int predict_impl(gpcc_fit_state* s, int NT, bool want_sd, bool want_cov, const double* d_extra, cudaStream_t st) {
    const int N = s->N, L = s->L;
    const auto& dp = s->p->pd[0].dp;
    cross_cov_kernel<KID><<<dim3((N + 255) / 256, std::min(NT, 32768)), 256, 0, st>>>(N, NT, dp.t, dp.band, s->tt.d, s->bandt.d, s->h, s->Z.d);
    trsm_lower_kernel<<<std::min((NT + TC - 1) / TC, 65535), 256, 0, st>>>(N, NT, s->Lc, s->Z.d);                 // Z = Lc^-1 k*
    col_stats_kernel<<<(NT + 7) / 8, 256, 0, st>>>(N, NT, L, s->Z.d, s->VU, s->w, s->bandt.d, s->h, s->postb_d, s->mu.d, s->R.d,
                                                  want_sd ? s->sd.d : nullptr);
    if (want_cov) {
        gemm_tn_kernel<<<dim3((NT + 63) / 64, (NT + 63) / 64), 256, 0, st>>>(NT, NT, N, s->Z.d, s->Z.d, s->G.d);   // Z'Z
        pred_cov_kernel<KID><<<dim3((NT + 255) / 256, std::min(NT, 32768)), 256, 0, st>>>(NT, L, s->G.d, s->R.d, s->tt.d, s->bandt.d, s->h,
                                                                                         s->postb_d, d_extra, s->S.d);
    }
    CUDA_TRY(cudaGetLastError());
    return 0;
}

int predict_common(gpcc_fit_state* s, const int* ntest_per_band, const double* ttest, const double* ytest,
                   const double* sigmatest, double* out_mu, double* out_sd, double* out_Sigma, double* out_ll, int* out_info) {
    if (!s) return fail(-1, "fit state is NULL");
    if (!ntest_per_band) return fail(-1, "NULL argument");
    const int L = s->L, N = s->N;
    long long NTl = 0;
    for (int l = 0; l < L; ++l) { if (ntest_per_band[l] < 0) return fail(-5, "negative test count"); NTl += ntest_per_band[l]; }
    if (NTl == 0) { if (out_ll) *out_ll = 0.0; if (out_info) *out_info = 0; return 0; }
    if (NTl > (1LL << 30) / std::max(1, N / 1024 + 1)) return fail(-7, "too many test points for one call");
    const int NT = (int)NTl;
    if (!ttest) return fail(-1, "NULL argument");
    std::vector<int> bandt(NT);
    for (int l = 0, k = 0; l < L; ++l) for (int i = 0; i < ntest_per_band[l]; ++i) bandt[k++] = l;
    DeviceState& ds = s->p->ctx->ds[0];
    CUDA_TRY(cudaSetDevice(s->dev));
    cudaStream_t st = ds.stream;
    const bool want_ll = out_ll != nullptr;
    const bool want_cov = out_Sigma || want_ll;
    CUDA_TRY(s->Z.reserve((size_t)N * NT));
    CUDA_TRY(s->R.reserve((size_t)L * NT));
    CUDA_TRY(s->mu.reserve(NT));
    CUDA_TRY(s->sd.reserve(NT));
    CUDA_TRY(s->tt.reserve(NT));
    CUDA_TRY(s->bandt.reserve(NT));
    if (want_cov) { CUDA_TRY(s->G.reserve((size_t)NT * NT)); CUDA_TRY(s->S.reserve((size_t)NT * NT)); }
    CUDA_TRY(cudaMemcpyAsync(s->tt.d, ttest, NT * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(s->bandt.d, bandt.data(), NT * sizeof(int), cudaMemcpyHostToDevice, st));
    std::vector<double> s2;
    if (want_ll) {
        s2.resize(NT);
        for (int i = 0; i < NT; ++i) s2[i] = sigmatest[i] * sigmatest[i];          // Sobs* (:317)
        CUDA_TRY(s->extra.reserve(NT)); CUDA_TRY(s->yv.reserve(NT)); CUDA_TRY(s->zv.reserve(NT));
        CUDA_TRY(s->scal.reserve(2 * GPCC_MAX_BANDS + 2)); CUDA_TRY(s->info.reserve(1));
        CUDA_TRY(cudaMemcpyAsync(s->extra.d, s2.data(), NT * sizeof(double), cudaMemcpyHostToDevice, st));
        CUDA_TRY(cudaMemcpyAsync(s->yv.d, ytest, NT * sizeof(double), cudaMemcpyHostToDevice, st));
    }
    int rc;
    const double* d_extra = want_ll ? s->extra.d : nullptr;
    switch (s->kernel_id) {
        case K_OU:  rc = predict_impl<K_OU>(s, NT, out_sd != nullptr, want_cov, d_extra, st); break;
        case K_RBF: rc = predict_impl<K_RBF>(s, NT, out_sd != nullptr, want_cov, d_extra, st); break;
        case K_M32: rc = predict_impl<K_M32>(s, NT, out_sd != nullptr, want_cov, d_extra, st); break;
        default:    rc = predict_impl<K_M52>(s, NT, out_sd != nullptr, want_cov, d_extra, st); break;
    }
    if (rc) return rc;
    ds.launches += want_cov ? 5 : 3;
    if (out_mu) CUDA_TRY(cudaMemcpyAsync(out_mu, s->mu.d, NT * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (out_sd) CUDA_TRY(cudaMemcpyAsync(out_sd, s->sd.d, NT * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (out_Sigma) CUDA_TRY(cudaMemcpyAsync(out_Sigma, s->S.d, (size_t)NT * NT * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (want_ll) {
        double* d_out = s->scal.d + 2 * GPCC_MAX_BANDS;
        chol_logpdf_kernel<<<1, 1024, 0, st>>>(NT, s->S.d, s->yv.d, s->mu.d, s->zv.d, d_out, s->info.d);
        CUDA_TRY(cudaGetLastError());
        int hinfo = 0;
        CUDA_TRY(cudaMemcpyAsync(out_ll, d_out, sizeof(double), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaMemcpyAsync(&hinfo, s->info.d, sizeof(int), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        if (out_info) *out_info = hinfo;
    }
    CUDA_TRY(cudaStreamSynchronize(st));
    return 0;
}

// one-entry cache behind the stateless entry points: repeated pred() calls at the same fitted hyper-parameters (the
// reference's closure usage, README.md:119-120) and postb + pred of one gpcc call share ONE factorisation
int cached_state(gpcc_problem* p, const double* delays, const double* alpha, double rho, gpcc_fit_state** out) {
    int rc = check_hyper(p, delays, alpha, rho);
    if (rc) return rc;
    gpcc_fit_state* c = p->cached_state;
    if (c && c->h.rho == rho && std::memcmp(c->h.delays, delays, p->L * sizeof(double)) == 0 &&
        std::memcmp(c->h.alpha, alpha, p->L * sizeof(double)) == 0) { *out = c; return 0; }
    if (c) { free_state(c); p->cached_state = nullptr; }
    rc = create_state(p, delays, alpha, rho, &c);
    if (rc) return rc;
    p->cached_state = c;
    *out = c;
    return 0;
}

}  // namespace

extern "C" {

int gpcc_fit_state_create(gpcc_problem* p, const double* delays, const double* alpha, double rho, gpcc_fit_state** out) {
    if (!out) return fail(-1, "out is NULL");
    *out = nullptr;
    int rc = check_hyper(p, delays, alpha, rho);
    if (rc) return rc;
    return create_state(p, delays, alpha, rho, out);
}

int gpcc_fit_state_destroy(gpcc_fit_state* s) {
    if (!s) return 0;
    if (s->p && s->p->cached_state == s) s->p->cached_state = nullptr;
    free_state(s);
    return 0;
}

int gpcc_fit_state_postb(const gpcc_fit_state* s, double* out_mu, double* out_Sigma) {
    if (!s || !out_mu || !out_Sigma) return fail(-1, "NULL argument");
    for (int l = 0; l < s->L; ++l) {
        out_mu[l] = s->postb_h.mu[l];
        for (int m = 0; m < s->L; ++m) out_Sigma[m * s->L + l] = s->postb_h.S[l][m];
    }
    return 0;
}

int gpcc_fit_state_predict(gpcc_fit_state* s, const int* ntest_per_band, const double* ttest, double* out_mu, double* out_sd,
                           double* out_Sigma) {
    return predict_common(s, ntest_per_band, ttest, nullptr, nullptr, out_mu, out_sd, out_Sigma, nullptr, nullptr);
}

int gpcc_fit_state_predict_loglik(gpcc_fit_state* s, const int* ntest_per_band, const double* ttest, const double* ytest,
                                  const double* sigmatest, double* out_ll, int* out_info) {
    if (!ytest || !sigmatest || !out_ll) return fail(-1, "NULL argument");
    return predict_common(s, ntest_per_band, ttest, ytest, sigmatest, nullptr, nullptr, nullptr, out_ll, out_info);
}

long long gpcc_fit_state_factorisations(const gpcc_fit_state* s) { return s ? s->n_factorisations : -1; }

int gpcc_fit_state_sample(gpcc_fit_state* s, unsigned long long seed, int nsamples, double* out_f, double* out_z) {
    if (!s || !out_f) return fail(-1, "NULL argument");
    if (nsamples < 1) return fail(-2, "nsamples < 1");
    const int N = s->N;
    const size_t n = (size_t)N * nsamples;
    DeviceState& ds = s->p->ctx->ds[0];
    CUDA_TRY(cudaSetDevice(s->dev));
    cudaStream_t st = ds.stream;
    CUDA_TRY(s->Z.reserve(n));          // deviates
    CUDA_TRY(s->G.reserve(n));          // draws
    normal_kernel<<<(int)std::min<size_t>(1184, (n / 2 + 255) / 256 + 1), 256, 0, st>>>(n, seed, s->Z.d);
    trmv_lower_kernel<<<dim3((N + 255) / 256, std::min((nsamples + 3) / 4, 1024)), 256, 0, st>>>(N, nsamples, s->Lc, s->Z.d, s->G.d);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(out_f, s->G.d, n * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (out_z) CUDA_TRY(cudaMemcpyAsync(out_z, s->Z.d, n * sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    ds.launches += 2;
    return 0;
}

int gpcc_postb(gpcc_problem* p, const double* delays, const double* alpha, double rho, double* out_mu, double* out_Sigma) {
    gpcc_fit_state* s = nullptr;
    int rc = cached_state(p, delays, alpha, rho, &s);
    if (rc) return rc;
    return gpcc_fit_state_postb(s, out_mu, out_Sigma);
}

int gpcc_predict(gpcc_problem* p, const double* delays, const double* alpha, double rho, const int* ntest_per_band,
                 const double* ttest, double* out_mu, double* out_sd, double* out_Sigma) {
    gpcc_fit_state* s = nullptr;
    int rc = cached_state(p, delays, alpha, rho, &s);
    if (rc) return rc;
    return gpcc_fit_state_predict(s, ntest_per_band, ttest, out_mu, out_sd, out_Sigma);
}

int gpcc_predict_loglik(gpcc_problem* p, const double* delays, const double* alpha, double rho, const int* ntest_per_band,
                        const double* ttest, const double* ytest, const double* sigmatest, double* out_ll, int* out_info) {
    gpcc_fit_state* s = nullptr;
    int rc = cached_state(p, delays, alpha, rho, &s);
    if (rc) return rc;
    return gpcc_fit_state_predict_loglik(s, ntest_per_band, ttest, ytest, sigmatest, out_ll, out_info);
}

}  // extern "C"
