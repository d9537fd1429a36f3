// Exact O(N) draws of the state-space model (gpcc_ss_sample): f ~ N(0, K + Sobs) for OU, matern32 and matern52, the draw
// of the reference's simulator (src/simulatedata.jl:128-145) without an N x N factor.
//
// Over the merged, delay-shifted times s_0 <= s_1 <= ... (the filter's order: smallest t - tau_l first, ties to the lower
// band, stable within a band) the f-state of the kernel's SDE is the affine recurrence
//   x_0 = C_0 w_0,  C_0 C_0' = P_inf;     x_k = A(D_k) x_(k-1) + C_k w_k,  C_k C_k' = Q(D_k),  D_k = s_k - s_(k-1)
// and the draw at merged step k, point i of band l, is f_i = alpha_l x_k[0] + sigma_i eps_i.  A and Q are the closed forms of
// ss_model.h; C_k is ss::noise_factor (D_k = 0 gives C_k = 0: a tie adds no process noise).
//
// Deviates: point i (input order) of sample s owns d process deviates (they drive the step that arrives at i) and one noise
// deviate, [s][i][d+1].  They come from the caller (z_in) or from Philox-4x32-10 with counter (i, sample0 + s, tag, call)
// and key = seed, two Box-Muller normals per call: a draw depends only on (seed, sample, i), not on the launch geometry, on
// nsamples or on the delays (common random numbers across delays).  gpcc_ss_sample uses the tag "SSMP" and sample0 = 0.
//
// The recurrence is a composition of affine maps (A_k, c_k = C_k w_k), evaluated as an inclusive scan per sample in three
// kernels with a fixed association, so every draw is bitwise reproducible:
//   1. ss_tile_kernel: one thread per (tile of TILE steps, sample) composes its tile into one map;
//   2. ss_scan_kernel: one CTA per sample scans the tile maps in chunks of SCAN (Hillis-Steele in shared memory, the carry
//      passed from chunk to chunk);
//   3. ss_rerun_kernel: every (tile, sample) thread re-runs its tile from its carry-in and writes f in input order.
// A_k and C_k are computed once per call (ss_step_kernel, one thread per step) and stored, d^2 + d(d+1)/2 + 2 doubles per
// step: phases 1 and 3 run once per sample, and a recomputation there would repeat ss::step and the factor nsamples x 2
// times.  Scratch is O(N) plus nsamples x tiles x d doubles of carries.
#include "gpcc_internal.h"
#include "kernfun.cuh"
#include "philox.cuh"
#include "ss_model.h"

namespace gpcc {
namespace {

constexpr int TILE = 64;                      // merged steps per tile (phases 1 and 3); fixed, so results never depend on the card
constexpr int SCAN = 256;                     // threads of the aggregate scan (phase 2)

template <int KID> struct Rec {               // layout of one stored step: A (d x d), packed lower C, alpha, sigma
    static constexpr int d = ss::Dim<KID>::d, NC = d * (d + 1) / 2, W = d * d + NC + 2;
};

__device__ __forceinline__ int band_of(const SSProblem& p, int j) {
    int l = 0;
    while (l + 1 < p.L && j >= p.band_start[l + 1]) ++l;
    return l;
}

// Points q of band m (sorted) with t_q - tau < s (incl = false) or <= s (incl = true): binary search within the band.
__device__ __forceinline__ int count_before(const SSProblem& p, int m, double tau, double s, bool incl) {
    const int a = p.band_start[m];
    int lo = a, hi = p.band_start[m + 1];
    while (lo < hi) {
        const int mid = lo + ((hi - lo) >> 1);
        const double v = p.t[mid] - tau;
        if (incl ? v <= s : v < s) lo = mid + 1;
        else hi = mid;
    }
    return lo - a;
}

// The first DD of the S = d + 1 deviates of point i of sample s.
template <int DD, int S>
__device__ __forceinline__ void deviates(const SSSampleArgs& a, int N, int s, int i, double (&w)[DD]) {
    if (a.zin) {
        const double* z = a.zin + ((size_t)s * N + i) * (size_t)S;
#pragma unroll
        for (int q = 0; q < DD; ++q) w[q] = z[q];
        return;
    }
    const uint2 key = make_uint2((unsigned)a.seed, (unsigned)(a.seed >> 32));
#pragma unroll
    for (int c = 0; 2 * c < DD; ++c) {
        const double2 g = box_muller(philox4x32_10(make_uint4((unsigned)i, (unsigned)(a.sample0 + s), a.tag, (unsigned)c), key));
        w[2 * c] = g.x;
        if (2 * c + 1 < DD) w[2 * c + 1] = g.y;
    }
}

// Merged position of sorted point j: its index within its band plus, for every other band m, the points with a smaller
// shifted time (ties: the points of lower bands come first).  Reproduces the filter's merge (statespace.cu).
__global__ void __launch_bounds__(256) ss_rank_kernel(SSProblem p, SSSampleArgs a, int* __restrict__ order) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= p.N) return;
    const int l = band_of(p, j);
    const double s = p.t[j] - a.tau[l];
    int rank = j - p.band_start[l];
    for (int m = 0; m < p.L; ++m)
        if (m != l) rank += count_before(p, m, a.tau[m], s, m < l);
    if (rank < p.N) order[rank] = j;
}

// A_k, C_k, alpha and sigma of merged step k (step 0: A = 0, C = chol(P_inf)), and the input index of its point.
template <int KID>
__global__ void __launch_bounds__(128) ss_step_kernel(SSProblem p, SSSampleArgs a, SSSampleScratch sc) {
    constexpr int d = ss::Dim<KID>::d, W = Rec<KID>::W;
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= p.N) return;
    const int j = sc.order[k];
    const int l = band_of(p, j);
    ss::Coef<d> c;
    ss::setup<KID>(a.rho, c);
    double A[d][d], C[d][d];
    if (k == 0) {
#pragma unroll
        for (int i = 0; i < d; ++i)
#pragma unroll
            for (int q = 0; q < d; ++q) A[i][q] = 0.0;
        ss::noise_factor<d>(c.Pinf, C);
    } else {
        const int jp = sc.order[k - 1];
        const double D = (p.t[j] - a.tau[l]) - (p.t[jp] - a.tau[band_of(p, jp)]);
        if (D > 0.0) {
            double Q[d][d], dA[d][d], dQ[d][d];
            ss::step<KID, false>(c, D, A, Q, dA, dQ);
            ss::noise_factor<d>(Q, C);
        } else {                                   // a tie: A = I, Q = 0 exactly
#pragma unroll
            for (int i = 0; i < d; ++i)
#pragma unroll
                for (int q = 0; q < d; ++q) { A[i][q] = i == q ? 1.0 : 0.0; C[i][q] = 0.0; }
        }
    }
    double* r = sc.step + (size_t)k * W;
#pragma unroll
    for (int i = 0; i < d; ++i)
#pragma unroll
        for (int q = 0; q < d; ++q) r[i * d + q] = A[i][q];
    int o = d * d;
#pragma unroll
    for (int i = 0; i < d; ++i)
#pragma unroll
        for (int q = 0; q <= i; ++q) r[o++] = C[i][q];
    r[W - 2] = a.alpha[l];
    r[W - 1] = sqrt(p.s2[j]);
    sc.idx[k] = a.perm[j];
}

// x = A x + C w for the stored step r
template <int KID>
__device__ __forceinline__ void advance(const double* __restrict__ r, const double (&w)[ss::Dim<KID>::d], double (&x)[ss::Dim<KID>::d]) {
    constexpr int d = ss::Dim<KID>::d;
    double y[d];
#pragma unroll
    for (int i = 0; i < d; ++i) {
        double s = 0.0;
#pragma unroll
        for (int q = 0; q < d; ++q) s = fma(r[i * d + q], x[q], s);
#pragma unroll
        for (int q = 0; q <= i; ++q) s = fma(r[d * d + i * (i + 1) / 2 + q], w[q], s);
        y[i] = s;
    }
#pragma unroll
    for (int i = 0; i < d; ++i) x[i] = y[i];
}

// Phase 1: the map of tile b for sample s, x -> M x + c (M only from sample 0: it does not depend on the deviates).
template <int KID>
__global__ void __launch_bounds__(128) ss_tile_kernel(int N, int tiles, SSSampleArgs a, SSSampleScratch sc) {
    constexpr int d = ss::Dim<KID>::d, W = Rec<KID>::W;
    const size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= (size_t)tiles * (size_t)a.nsamples) return;
    const int b = (int)(g % (size_t)tiles), s = (int)(g / (size_t)tiles);
    const int k0 = b * TILE, k1 = min(N, k0 + TILE);
    double x[d], M[d][d];
#pragma unroll
    for (int i = 0; i < d; ++i) {
        x[i] = 0.0;
#pragma unroll
        for (int q = 0; q < d; ++q) M[i][q] = i == q ? 1.0 : 0.0;
    }
    for (int k = k0; k < k1; ++k) {
        const double* r = sc.step + (size_t)k * W;
        double w[d];
        deviates<d, d + 1>(a, N, s, sc.idx[k], w);
        advance<KID>(r, w, x);
        if (s == 0) {
            double T[d][d];
#pragma unroll
            for (int i = 0; i < d; ++i)
#pragma unroll
                for (int q = 0; q < d; ++q) {
                    double v = 0.0;
#pragma unroll
                    for (int u = 0; u < d; ++u) v = fma(r[i * d + u], M[u][q], v);
                    T[i][q] = v;
                }
#pragma unroll
            for (int i = 0; i < d; ++i)
#pragma unroll
                for (int q = 0; q < d; ++q) M[i][q] = T[i][q];
        }
    }
#pragma unroll
    for (int i = 0; i < d; ++i) sc.aggc[((size_t)s * tiles + b) * d + i] = x[i];
    if (s == 0) {
#pragma unroll
        for (int i = 0; i < d; ++i)
#pragma unroll
            for (int q = 0; q < d; ++q) sc.aggA[(size_t)b * d * d + i * d + q] = M[i][q];
    }
}

// Phase 2: one CTA per sample.  Inclusive scan of the tile maps, SCAN tiles at a time; aggc[s][b] becomes the state after
// tile b.  Tile 0 holds step 0 (A = 0), so every prefix map is constant and its value is that state.
template <int KID>
__global__ void __launch_bounds__(SCAN) ss_scan_kernel(int tiles, SSSampleScratch sc) {
    constexpr int d = ss::Dim<KID>::d;
    __shared__ double shA[SCAN][d * d], shc[SCAN][d];
    const int s = blockIdx.x, tid = threadIdx.x;
    double carry[d];
#pragma unroll
    for (int i = 0; i < d; ++i) carry[i] = 0.0;
    for (int c0 = 0; c0 < tiles; c0 += SCAN) {
        const int b = c0 + tid;
        double A[d][d], c[d];
#pragma unroll
        for (int i = 0; i < d; ++i) {
            c[i] = b < tiles ? sc.aggc[((size_t)s * tiles + b) * d + i] : 0.0;
#pragma unroll
            for (int q = 0; q < d; ++q) A[i][q] = b < tiles ? sc.aggA[(size_t)b * d * d + i * d + q] : (i == q ? 1.0 : 0.0);
        }
        for (int off = 1; off < SCAN; off <<= 1) {
#pragma unroll
            for (int i = 0; i < d; ++i) {
                shc[tid][i] = c[i];
#pragma unroll
                for (int q = 0; q < d; ++q) shA[tid][i * d + q] = A[i][q];
            }
            __syncthreads();
            if (tid >= off) {                        // (A, c) o (A', c') = (A A', A c' + c), (A', c') the earlier range
                const int o = tid - off;
                double nA[d][d], nc[d];
#pragma unroll
                for (int i = 0; i < d; ++i) {
                    double v = c[i];
#pragma unroll
                    for (int u = 0; u < d; ++u) v = fma(A[i][u], shc[o][u], v);
                    nc[i] = v;
#pragma unroll
                    for (int q = 0; q < d; ++q) {
                        double t = 0.0;
#pragma unroll
                        for (int u = 0; u < d; ++u) t = fma(A[i][u], shA[o][u * d + q], t);
                        nA[i][q] = t;
                    }
                }
#pragma unroll
                for (int i = 0; i < d; ++i) {
                    c[i] = nc[i];
#pragma unroll
                    for (int q = 0; q < d; ++q) A[i][q] = nA[i][q];
                }
            }
            __syncthreads();
        }
        double x[d];
#pragma unroll
        for (int i = 0; i < d; ++i) {
            double v = c[i];
#pragma unroll
            for (int u = 0; u < d; ++u) v = fma(A[i][u], carry[u], v);
            x[i] = v;
        }
        if (b < tiles) {
#pragma unroll
            for (int i = 0; i < d; ++i) sc.aggc[((size_t)s * tiles + b) * d + i] = x[i];
        }
        if (tid == SCAN - 1) {
#pragma unroll
            for (int i = 0; i < d; ++i) shc[0][i] = x[i];
        }
        __syncthreads();
#pragma unroll
        for (int i = 0; i < d; ++i) carry[i] = shc[0][i];
        __syncthreads();
    }
}

// Phase 3: tile b of sample s again, from the state after tile b-1; f and (optionally) the deviates in input order.
template <int KID>
__global__ void __launch_bounds__(128) ss_rerun_kernel(int N, int tiles, SSSampleArgs a, SSSampleScratch sc) {
    constexpr int d = ss::Dim<KID>::d, W = Rec<KID>::W;
    const size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= (size_t)tiles * (size_t)a.nsamples) return;
    const int b = (int)(g % (size_t)tiles), s = (int)(g / (size_t)tiles);
    const int k0 = b * TILE, k1 = min(N, k0 + TILE);
    double x[d];
#pragma unroll
    for (int i = 0; i < d; ++i) x[i] = b > 0 ? sc.aggc[((size_t)s * tiles + b - 1) * d + i] : 0.0;
    for (int k = k0; k < k1; ++k) {
        const double* r = sc.step + (size_t)k * W;
        const int i = sc.idx[k];
        double z[d + 1], w[d];
        deviates<d + 1, d + 1>(a, N, s, i, z);
#pragma unroll
        for (int q = 0; q < d; ++q) w[q] = z[q];
        advance<KID>(r, w, x);
        const size_t o = (size_t)s * N + i;
        a.f[o] = fma(r[W - 2], x[0], r[W - 1] * z[d]);
        if (a.zout) {
#pragma unroll
            for (int q = 0; q <= d; ++q) a.zout[o * (d + 1) + q] = z[q];
        }
    }
}

template <int KID>
cudaError_t launch(const SSProblem& p, const SSSampleArgs& a, const SSSampleScratch& s, cudaStream_t st) {
    const int N = p.N, tiles = (N + TILE - 1) / TILE;
    const size_t blocks = ((size_t)tiles * (size_t)a.nsamples + 127) / 128;
    if (blocks > 0x7fffffffu) return cudaErrorInvalidValue;
    ss_rank_kernel<<<(N + 255) / 256, 256, 0, st>>>(p, a, s.order);
    ss_step_kernel<KID><<<(N + 127) / 128, 128, 0, st>>>(p, a, s);
    ss_tile_kernel<KID><<<(unsigned)blocks, 128, 0, st>>>(N, tiles, a, s);
    ss_scan_kernel<KID><<<a.nsamples, SCAN, 0, st>>>(tiles, s);
    ss_rerun_kernel<KID><<<(unsigned)blocks, 128, 0, st>>>(N, tiles, a, s);
    return cudaGetLastError();
}

int state_dim(int kernel_id) { return kernel_id == K_OU ? 1 : kernel_id == K_M32 ? 2 : 3; }

}  // namespace

cudaError_t statespace_rank_launch(const SSProblem& p, const double* tau, int* order, cudaStream_t stream) {
    if (p.N <= 0) return cudaSuccess;
    SSSampleArgs a;
    for (int l = 0; l < p.L; ++l) a.tau[l] = tau[l];
    ss_rank_kernel<<<(p.N + 255) / 256, 256, 0, stream>>>(p, a, order);
    return cudaGetLastError();
}

void statespace_sample_scratch(int kernel_id, int N, int nsamples, size_t& n_step, size_t& n_aggA, size_t& n_aggc) {
    const size_t d = (size_t)state_dim(kernel_id), tiles = ((size_t)N + TILE - 1) / TILE;
    n_step = (size_t)N * (d * d + d * (d + 1) / 2 + 2);
    n_aggA = tiles * d * d;
    n_aggc = (size_t)nsamples * tiles * d;
}

cudaError_t statespace_sample_launch(int kernel_id, const SSProblem& p, const SSSampleArgs& a, const SSSampleScratch& s,
                                     cudaStream_t stream) {
    if (p.N <= 0 || a.nsamples <= 0) return cudaErrorInvalidValue;
    switch (kernel_id) {
        case K_OU:  return launch<K_OU>(p, a, s, stream);
        case K_M32: return launch<K_M32>(p, a, s, stream);
        case K_M52: return launch<K_M52>(p, a, s, stream);
        default:    return cudaErrorInvalidValue;     // rbf: rejected by gpcc_problem_set_method
    }
}

}  // namespace gpcc
