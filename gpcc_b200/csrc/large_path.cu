// Large-N path: the matrix lives in HBM in a tile layout, factorised / inverted by a blocked symmetric sweep whose
// flops run on the FP64 tensor pipe (DMMA.8x8x4 = mma.sync.m8n8k4.f64; tcgen05 has no f64 kind).
//
// Replaces, for N too large for the register-resident kernel, the same reference code as small_sweep.cu:
//   K = delayedCovariance(...) + Sobs + B ; logpdf(MvNormal(bbar, K), Y)      (gpccfixdelay_marginaliseb.jl:133-141)
// plus K^-1 for the analytic gradient (north_star).
//
// Data layout (per matrix, lower triangle only):  macro tiles 128x128, tile (I,J), I>=J at index I(I+1)/2+J, each a
// 16x16 grid of 8x8 micro tiles stored row-major -- exactly the DMMA accumulator fragment (lane t owns elements
// 2t, 2t+1 of a micro tile), so every global access of the GEMM kernels is a fully coalesced 512-byte warp
// transaction.  Panels (N x 128 operands) are stored as [k/4][row/8][8 rows x 4 k] chunks = the DMMA A/B fragment,
// contiguous 16 KB per 16-wide K slice, so they are staged into shared memory with cp.async.bulk (TMA bulk copy
// engine) completing on an mbarrier, and read back with conflict-free LDS.64.
//
// Algorithm, block step k = 0..T-1 (pivot block D = A_kk, 128x128):
//   pivot   : D = L L' (in shared memory), Linv = L^-1, logdet += 2 sum log L_jj, z = Linv r_k, quad += z'z;
//             sweep mode also Dinv = Linv' Linv, A_kk <- -Dinv, r_k <- Linv' z.
//   gather  : column k of the symmetric matrix -> panel layout P (tiles (I,k), I>k and (k,I)' for I<k)
//   panel   : X = P Linv'   (DMMA)  -> panel layout;  r_I -= X_I z;   sweep mode also Q = P Dinv -> written back as
//             column k;  forward mode writes X back (the matrix then holds the Cholesky factor).
//   update  : A_IJ -= X_I X_J'  (DMMA) for all lower tiles with I,J != k (sweep) or I,J > k (forward = Cholesky).
// Forward mode is exactly a right-looking blocked Cholesky (N^3/3 flop); sweep mode continues the elimination over
// the already-processed part and leaves -A^-1 (N^3 flop, the same as potrf+potri) with a = A^-1 r in r.
#include "gpcc_internal.h"
#include "kernfun.cuh"
#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdint>
#include <cstdlib>
#include <vector>
#include <cstdio>
#include <cstring>
#include <map>
#include <memory>

namespace gpcc {
namespace {

constexpr int BT = 128;            // macro tile edge
constexpr int TILE_ELEMS = BT * BT;
constexpr int KCH = 16;            // K slice staged per pipeline stage
constexpr int NCHUNK = BT / KCH;   // 8
constexpr int STAGES = 3;
constexpr int CHUNK_ELEMS = KCH * BT;           // 2048 doubles = 16 KB per operand per stage
constexpr double LOG2PI = 1.8378770664093454835606594728112;

__host__ __device__ __forceinline__ size_t tile_index(int I, int J) { return (size_t)I * (I + 1) / 2 + J; }
// element (r,c) inside a macro tile (tile layout)
__device__ __forceinline__ int tl_off(int r, int c) { return (((r >> 3) * 16 + (c >> 3)) << 6) + ((r & 7) << 3) + (c & 7); }
// element (row r, k index c) inside a 128x128 panel block (panel layout)
__device__ __forceinline__ int pl_off(int r, int c) { return (((c >> 2) * 16 + (r >> 3)) << 5) + ((r & 7) << 2) + (c & 3); }

struct LargeArgs {
    int N, L, T, Np, kid;
    int sweep;          // 1: full symmetric sweep (inverse, gradient); 0: forward only (Cholesky, logL)
    int Tp;             // > 0 (forward mode only): the first Tp block rows / columns are IDENTICAL in all matrices of the wave
                        // (same hyper-parameters, same delays of all bands but the last): matrix 0 computes them for everybody
    int mode_postb;
    double* mats;       // [B][ntiles][TILE_ELEMS]
    double* Pws;        // [B][T][TILE_ELEMS]   gathered column, panel layout
    double* Xws;        // [B][T][TILE_ELEMS]   X = P Linv', panel layout
    double* Linv;       // [B][TILE_ELEMS]      Linv[c][k], panel layout
    double* Dinv;       // [B][TILE_ELEMS]      Dinv[c][k], panel layout
    double* rvec;       // [B][Np]
    double* zk;         // [B][BT]
    double* scal;       // [B][4]  logdet, quad
    int* info;          // [B]
    double* tsh;        // [B][Np] shifted times
    double* av;         // [B][Np] alpha per point (0 on padding)
    double* part;       // [B][T][T][BT] gradient row-sum partials
    double* epart;      // [B][ntiles]
    size_t mat_stride;  // doubles per matrix
    size_t x_parity_stride;   // Xws is double buffered by step parity (look-ahead: update k still reads X_k while panel k+1 writes)
    // Last-band cache (forward mode, three or more bands; see large_eval).  Pivots k < Tq lie in band 1,
    // block rows I >= Tc in the last band.  What steps k < Tq do to the last band's rows -- the panels X_I^(k), the state of block
    // (3,3) and of r_3 after step Tq-1 -- depends on the LAST delay only: cmode 1 (FILL) computes it once per distinct value and
    // exports it to slot[m]; cmode 2 (USE) imports it instead of recomputing it for every candidate.
    int Tq, Tc, cmode;
    const int* eidx;    // [B] evaluation index of matrix m (nullptr: e0 + m)
    const int* slot;    // [B] cache slot of matrix m
    double *XC, *AC, *RC;
    size_t xc_stride, ac_stride, rc_stride;   // doubles per slot
};
__device__ __forceinline__ double* xc_tile(const LargeArgs& a, int m, int k, int I) {
    return a.XC + (size_t)a.slot[m] * a.xc_stride + ((size_t)k * (a.T - a.Tc) + (I - a.Tc)) * TILE_ELEMS;
}
__device__ __forceinline__ double* ac_tile(const LargeArgs& a, int m, int I, int J) {
    return a.AC + (size_t)a.slot[m] * a.ac_stride + tile_index(I - a.Tc, J - a.Tc) * TILE_ELEMS;
}
// FILL never touches the middle band; USE leaves the last band's rows alone while the pivot is in band 1
__device__ __forceinline__ bool cache_skips_row(const LargeArgs& a, int k, int I) {
    return (a.cmode == 1 && I >= a.Tq && I < a.Tc) || (a.cmode == 2 && k < a.Tq && I >= a.Tc);
}

// ---------------------------------------------------------------------------------------------------------------
// PTX helpers: mbarrier + bulk async copy (TMA engine, 1-D), DMMA
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE;\n"
        "bra WAIT_LOOP;\n"
        "DONE:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

// ---------------------------------------------------------------------------------------------------------------
// 128x128x128 DMMA main loop of the panel kernel.
// acc += A B',  A and B are 128x128 panel-layout blocks in global memory (contiguous 16 KB per K slice).
// 8 warps; warp w owns rows 32*(w&3).., cols 64*(w>>2)..  -> acc[4][8][2] per lane.
// ---------------------------------------------------------------------------------------------------------------
struct GemmSmem {
    double a[STAGES][CHUNK_ELEMS];
    double b[STAGES][CHUNK_ELEMS];
    uint64_t full[STAGES];
};

__device__ __forceinline__ void gemm_mainloop(GemmSmem& sm, const double* __restrict__ gA, const double* __restrict__ gB,
                                              double (&acc)[4][8][2]) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int ro0 = (warp & 3) * 4, co0 = (warp >> 2) * 8;
    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) mbar_init(&sm.full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_expect_tx(&sm.full[s], 2 * CHUNK_ELEMS * sizeof(double));
            bulk_g2s(sm.a[s], gA + (size_t)s * CHUNK_ELEMS, CHUNK_ELEMS * sizeof(double), &sm.full[s]);
            bulk_g2s(sm.b[s], gB + (size_t)s * CHUNK_ELEMS, CHUNK_ELEMS * sizeof(double), &sm.full[s]);
        }
    }
#pragma unroll 1
    for (int ch = 0; ch < NCHUNK; ++ch) {
        const int s = ch % STAGES;
        mbar_wait(&sm.full[s], (ch / STAGES) & 1);
        const double* sa = sm.a[s];
        const double* sb = sm.b[s];
#pragma unroll
        for (int k4 = 0; k4 < KCH / 4; ++k4) {
            double a[4], b[8];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = sa[((k4 * 16 + ro0 + i) << 5) + lane];
#pragma unroll
            for (int j = 0; j < 8; ++j) b[j] = sb[((k4 * 16 + co0 + j) << 5) + lane];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) dmma(acc[i][j][0], acc[i][j][1], a[i], b[j]);
        }
        __syncthreads();   // everyone is done with stage s
        if (tid == 0 && ch + STAGES < NCHUNK) {
            mbar_expect_tx(&sm.full[s], 2 * CHUNK_ELEMS * sizeof(double));
            bulk_g2s(sm.a[s], gA + (size_t)(ch + STAGES) * CHUNK_ELEMS, CHUNK_ELEMS * sizeof(double), &sm.full[s]);
            bulk_g2s(sm.b[s], gB + (size_t)(ch + STAGES) * CHUNK_ELEMS, CHUNK_ELEMS * sizeof(double), &sm.full[s]);
        }
    }
}

// Half-tile form of the main loop for the trailing update: 4 warps compute the 128 x 64 column half `h` of a tile (warp w: rows
// 32 w.., all 64 columns).  164 registers x 128 threads and 72 KB of staging let THREE such CTAs share an SM, so the global
// load / store of one CTA's accumulators (the C tile: 131 KB per tile and step, not overlapped inside a CTA) hides under the
// DMMAs of the others, and every scheduler holds three warps instead of two.
struct GemmSmemHalf {
    double a[STAGES][CHUNK_ELEMS];
    double b[STAGES][CHUNK_ELEMS / 2];
    uint64_t full[STAGES];
};

__device__ __forceinline__ void stage_half(GemmSmemHalf& sm, int s, const double* gA, const double* gB, int ch, int h) {
    mbar_expect_tx(&sm.full[s], (CHUNK_ELEMS + CHUNK_ELEMS / 2) * sizeof(double));
    bulk_g2s(sm.a[s], gA + (size_t)ch * CHUNK_ELEMS, CHUNK_ELEMS * sizeof(double), &sm.full[s]);
#pragma unroll
    for (int k4 = 0; k4 < KCH / 4; ++k4)      // the column half is 8 of the 16 row groups of every 4-deep slice: 2 KB each
        bulk_g2s(sm.b[s] + k4 * 256, gB + (size_t)ch * CHUNK_ELEMS + (size_t)(k4 * 16 + 8 * h) * 32, 256 * sizeof(double), &sm.full[s]);
}

__device__ __forceinline__ void gemm_mainloop_half(GemmSmemHalf& sm, const double* __restrict__ gA, const double* __restrict__ gB, int h,
                                                   double (&acc)[4][8][2]) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int ro0 = warp * 4;
    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) mbar_init(&sm.full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0)
        for (int s = 0; s < STAGES; ++s) stage_half(sm, s, gA, gB, s, h);
#pragma unroll 1
    for (int ch = 0; ch < NCHUNK; ++ch) {
        const int s = ch % STAGES;
        mbar_wait(&sm.full[s], (ch / STAGES) & 1);
        const double* sa = sm.a[s];
        const double* sb = sm.b[s];
#pragma unroll
        for (int k4 = 0; k4 < KCH / 4; ++k4) {
            double av[4], bv[8];
#pragma unroll
            for (int i = 0; i < 4; ++i) av[i] = -sa[((k4 * 16 + ro0 + i) << 5) + lane];
#pragma unroll
            for (int j = 0; j < 8; ++j) bv[j] = sb[((k4 * 8 + j) << 5) + lane];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) dmma(acc[i][j][0], acc[i][j][1], av[i], bv[j]);
        }
        __syncthreads();   // everyone is done with stage s
        if (tid == 0 && ch + STAGES < NCHUNK) stage_half(sm, s, gA, gB, ch + STAGES, h);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// prep: shifted times, per-point alpha, right-hand side
// ---------------------------------------------------------------------------------------------------------------
__global__ void prep_kernel(DevProblem p, EvalBatch b, int e0, LargeArgs a) {
    const int m = blockIdx.y, e = a.eidx ? a.eidx[m] : e0 + m;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < a.Np; i += gridDim.x * blockDim.x) {
        double ts = 0.0, al = 0.0, r = 0.0;
        if (i < a.N) {
            const int bi = p.band[i];
            ts = p.t[i] - b.delays[(size_t)e * a.L + bi];     // delayedCovariance.jl:27
            al = b.alpha[(size_t)e * a.L + bi];
            r = a.mode_postb ? p.y[i] : p.resid[i];
        }
        if (a.cmode == 2 && i >= a.Tc * BT) r = a.RC[(size_t)a.slot[m] * a.rc_stride + (i - a.Tc * BT)];   // r_3 after step Tq-1
        a.tsh[(size_t)m * a.Np + i] = ts;
        a.av[(size_t)m * a.Np + i] = al;
        a.rvec[(size_t)m * a.Np + i] = r;
    }
    if (blockIdx.x == 0 && threadIdx.x < 4) a.scal[(size_t)m * 4 + threadIdx.x] = 0.0;
    if (blockIdx.x == 0 && threadIdx.x == 0) a.info[m] = 0;
}

// ---------------------------------------------------------------------------------------------------------------
// K1: covariance assembly into the tile layout (HBM-write bound: 4 N (N+1) bytes of unique output per matrix).
// One CTA per lower macro tile; the 128 row times and 128 column times are staged in shared memory; every warp
// store is one coalesced 512-byte micro tile (16-byte vector stores).
// ---------------------------------------------------------------------------------------------------------------
template <int KID>
__global__ void __launch_bounds__(256) assemble_kernel(DevProblem p, EvalBatch b, int e0, LargeArgs a) {
    __shared__ double tr[BT], tc[BT], ar[BT], ac[BT], dr[BT], sr[BT];
    __shared__ int br[BT], bc[BT];
    const int m = blockIdx.y, e = a.eidx ? a.eidx[m] : e0 + m;
    // decode lower tile index
    const int tix = blockIdx.x;
    int I = (int)((sqrtf(8.0f * (float)tix + 1.0f) - 1.0f) * 0.5f);
    while ((size_t)I * (I + 1) / 2 > (size_t)tix) --I;
    while ((size_t)(I + 1) * (I + 2) / 2 <= (size_t)tix) ++I;
    const int J = tix - I * (I + 1) / 2;
    if (a.Tp && m > 0 && I < a.Tp) return;        // shared prefix tile: assembled (and factorised) once, by matrix 0
    const int tid = threadIdx.x;
    if (a.cmode == 1 && ((I >= a.Tq && I < a.Tc) || (J >= a.Tq && J < a.Tc))) return;   // FILL: nothing of the middle band
    if (a.cmode == 2 && I >= a.Tc) {
        if (J < a.Tq) return;                     // block (3,1) is only ever read by the cached steps
        if (J >= a.Tc) {                          // block (3,3) as steps 0 .. Tq-1 leave it
            const double2* src = reinterpret_cast<const double2*>(ac_tile(a, m, I, J));
            double2* dst = reinterpret_cast<double2*>(a.mats + (size_t)m * a.mat_stride + tile_index(I, J) * TILE_ELEMS);
            for (int q = tid; q < TILE_ELEMS / 2; q += 256) dst[q] = src[q];
            return;
        }
    }
    if (tid < BT) {
        const int i = I * BT + tid;
        tr[tid] = a.tsh[(size_t)m * a.Np + i];
        ar[tid] = a.av[(size_t)m * a.Np + i];
        dr[tid] = i < a.N ? p.s2[i] : 0.0;
        sr[tid] = (i < a.N && !a.mode_postb) ? p.sigb[i] : 0.0;
        br[tid] = i < a.N ? p.band[i] : -1 - i;
    } else {
        const int c = tid - BT, j = J * BT + c;
        tc[c] = a.tsh[(size_t)m * a.Np + j];
        ac[c] = a.av[(size_t)m * a.Np + j];
        bc[c] = j < a.N ? p.band[j] : -1 - j;
    }
    __syncthreads();
    const KernParams kp = make_kern_params(KID, b.rho[e]);
    double* tile = a.mats + (size_t)m * a.mat_stride + tile_index(I, J) * TILE_ELEMS;
    const int lane = tid & 31, warp = tid >> 5;
    const int rr = lane >> 2, cc = (lane & 3) * 2;
    for (int mt = warp; mt < 256; mt += 8) {       // micro tile (mi, mj)
        const int mi = mt >> 4, mj = mt & 15;
        const int r = mi * 8 + rr, c = mj * 8 + cc;
        const int gi = I * BT + r;
        double v[2];
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const int gj = J * BT + c + q;
            double val = (ar[r] * ac[c + q]) * kern_value<KID>(tr[r] - tc[c + q], kp);   // delayedCovariance.jl:27
            if (gi == gj) val += dr[r];                                                      // + Sobs (:135)
            if (br[r] == bc[c + q]) val += sr[r];                                            // + B
            if (gi >= a.N && gi == gj) val = 1.0;                                            // identity on the padding
            v[q] = val;
        }
        *reinterpret_cast<double2*>(tile + (mt << 6) + 2 * lane) = make_double2(v[0], v[1]);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// pivot: Cholesky + triangular inverse of the 128x128 diagonal block in shared memory (one CTA per matrix).
// S is column-major with leading dimension 129 (conflict-free along rows and columns).
// ---------------------------------------------------------------------------------------------------------------
constexpr int PLD = BT + 1;
__device__ __forceinline__ double& SE(double* S, int i, int j) { return S[j * PLD + i]; }

__global__ void __launch_bounds__(256) pivot_kernel(LargeArgs a, int k) {
    extern __shared__ double sh[];
    double* S = sh;                    // [BT][PLD]
    double* zz = S + BT * PLD;         // [BT]
    double* rk = zz + BT;              // [BT]
    double* ldiag = rk + BT;           // [BT] diagonal of L
    __shared__ int s_bad;
    const int m = blockIdx.x, tid = threadIdx.x;
    if (a.Tp && k < a.Tp && m > 0) return;         // shared prefix: matrix 0 factorises the diagonal block for the whole wave
    const int ty = tid >> 4, tx = tid & 15;
    double* tile = a.mats + (size_t)m * a.mat_stride + tile_index(k, k) * TILE_ELEMS;
    for (int e = tid; e < BT * BT / 2; e += 256) {           // coalesced double2 reads of the tile layout
        const double2 v = *reinterpret_cast<const double2*>(tile + 2 * e);
        const int mt = e >> 5, w = e & 31;
        const int r = (mt >> 4) * 8 + (w >> 2), c = (mt & 15) * 8 + (w & 3) * 2;
        SE(S, r, c) = (c <= r) ? v.x : 0.0;
        SE(S, r, c + 1) = (c + 1 <= r) ? v.y : 0.0;
    }
    if (tid < BT) rk[tid] = a.rvec[(size_t)m * a.Np + k * BT + tid];
    if (tid == 0) s_bad = 0;
    __syncthreads();
#ifdef GPCC_PIVOT_PROF
    long long tp0 = clock64();
#endif
    // ---- blocked Cholesky, panels of NB = 16 columns -----------------------------------------------------------------------
    // Inside a panel the columns are formed LEFT-LOOKING, one thread per row: column j first receives the updates of the
    // panel columns before it (a dot product of <= 15 terms per row; every thread also forms the pivot itself, with the same
    // operations, so that no broadcast is needed), is scaled, and ONE barrier publishes it.  Behind the panel: one rank-16
    // update of everything to its right, 4 x 4 register blocks per thread, 16 FMAs per 8 shared-memory loads.
    // History (profiles/README.md, round 2): the unblocked form (rank-1 update of the whole trailing block after every column,
    // 2 barriers per column) took ~330 us of a 536 us kernel that is the critical path of every block step; a right-looking
    // panel 79 us; this form is measured there as well.
    constexpr int NB = 16;
    for (int j0 = 0; j0 < BT; j0 += NB) {
        for (int j = j0; j < j0 + NB; ++j) {
            if (tid >= j && tid < BT) {
                const int i = tid;
                // all loads first (predicated off beyond column j), then two short FMA chains per sum: the loop form
                // (load, load, fma, fma per term) ran at one shared-memory round trip per term
                double lik[NB], ljk[NB];
#pragma unroll
                for (int q = 0; q < NB; ++q) {
                    const bool on = j0 + q < j;
                    lik[q] = on ? SE(S, i, j0 + q) : 0.0;
                    ljk[q] = on ? SE(S, j, j0 + q) : 0.0;
                }
                double s0 = SE(S, i, j), s1 = 0.0, d0 = SE(S, j, j), d1 = 0.0;
#pragma unroll
                for (int q = 0; q < NB; q += 2) {
                    s0 = fma(-lik[q], ljk[q], s0);
                    s1 = fma(-lik[q + 1], ljk[q + 1], s1);
                    d0 = fma(-ljk[q], ljk[q], d0);
                    d1 = fma(-ljk[q + 1], ljk[q + 1], d1);
                }
                const double sij = s0 + s1, sjj = d0 + d1;
                const double rs = rsqrt(sjj);                   // NaN for a non-positive pivot, like sqrt
                const double sq = sjj * rs;
                if (i == j) {                                   // S(j,j) itself is written after the panel: the other rows still read it
                    ldiag[j] = sq;
                    if (!(sjj > 0.0) && s_bad == 0) s_bad = j + 1;
                } else {
                    SE(S, i, j) = sij * rs;
                }
            }
            __syncthreads();
        }
        if (tid >= j0 && tid < j0 + NB) SE(S, tid, tid) = ldiag[tid];
        __syncthreads();
        const int r0 = j0 + NB;                                // trailing block starts here
        const int nbk = (BT - r0) / 4;                         // 4 x 4 register blocks per side
        const int nblk = nbk * (nbk + 1) / 2;
        for (int blk = tid; blk < nblk; blk += 256) {
            int bi = (int)((sqrtf(8.0f * (float)blk + 1.0f) - 1.0f) * 0.5f);
            while (bi * (bi + 1) / 2 > blk) --bi;
            while ((bi + 1) * (bi + 2) / 2 <= blk) ++bi;
            const int bj = blk - bi * (bi + 1) / 2;
            const int i0 = r0 + 4 * bi, c0 = r0 + 4 * bj;
            double acc[4][4];
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int q = 0; q < 4; ++q) acc[r][q] = 0.0;
#pragma unroll 4
            for (int kk = j0; kk < j0 + NB; ++kk) {
                double li[4], lc[4];
#pragma unroll
                for (int r = 0; r < 4; ++r) { li[r] = SE(S, i0 + r, kk); lc[r] = SE(S, c0 + r, kk); }
#pragma unroll
                for (int r = 0; r < 4; ++r)
#pragma unroll
                    for (int q = 0; q < 4; ++q) acc[r][q] = fma(li[r], lc[q], acc[r][q]);
            }
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    if (i0 + r >= c0 + q) SE(S, i0 + r, c0 + q) -= acc[r][q];      // lower triangle only: the upper part stays zero
        }
        __syncthreads();                                       // the next panel reads what the trailing update wrote
    }
    __syncthreads();
#ifdef GPCC_PIVOT_PROF
    long long tp1 = clock64();
#endif
    if (!a.sweep) {   // forward mode: the diagonal tile keeps the Cholesky factor (upper part zero)
        for (int e = tid; e < BT * BT / 2; e += 256) {
            const int mt = e >> 5, w = e & 31;
            const int r = (mt >> 4) * 8 + (w >> 2), c = (mt & 15) * 8 + (w & 3) * 2;
            *reinterpret_cast<double2*>(tile + 2 * e) = make_double2(SE(S, r, c), SE(S, r, c + 1));
        }
    }
    // ---- in-place inverse of the lower-triangular factor, blocked (LAPACK dtrtri 'L': last block column first) ----------
    //   A21 <- -Linv22 A21 inv(A11),  A11 <- inv(A11)        with 16-column blocks.
    // Linv22 A21 (the bulk: R^2/2 x 16 FMAs) runs on warps 0-6 in 2 x 4 register blocks into a staging buffer while warp 7
    // inverts the 16 x 16 diagonal block (one lane per column, forward substitution in registers); then the staging buffer
    // is multiplied by the block inverse.  The unblocked form (dtrti2: two threads per row, 2 barriers per column, dot
    // products of up to 127 terms) took 107 us of the kernel.
    {
        double* Tb = zz + 3 * BT;            // [<=112][16] staging of Linv22 A21 (row-major, stride 17)
        double* Db = Tb + 112 * 17;          // [16][17] inverse of the diagonal block (row-major)
        const int lane = tid & 31, warp = tid >> 5;
        for (int j0 = BT - NB; j0 >= 0; j0 -= NB) {
            const int r0 = j0 + NB, R = BT - r0;
            if (warp == 7) {
                if (lane < NB) {             // column c = lane of inv(A11): x_r = (delta_rc - sum_{q<r} A11(r,q) x_q) / A11(r,r)
                    const int c = lane;
                    double x[NB];
#pragma unroll
                    for (int r = 0; r < NB; ++r) {
                        double acc = (r == c) ? 1.0 : 0.0;
#pragma unroll
                        for (int q = 0; q < NB; ++q)
                            if (q < r) acc = fma(-SE(S, j0 + r, j0 + q), x[q], acc);
                        x[r] = (r >= c) ? acc / SE(S, j0 + r, j0 + r) : 0.0;
                    }
#pragma unroll
                    for (int r = 0; r < NB; ++r) Db[r * 17 + c] = x[r];
                }
            } else {
                // Tb(i, c) = sum_{q = r0..i} Linv22(i, q) A21(q, c), i in [r0, BT), c in [0, 16): 2 rows x 4 columns per thread
                const int nrb = R / 2;                     // R is a multiple of 16
                for (int blk = tid; blk < nrb * 4; blk += 224) {
                    const int ib = blk >> 2, cb = blk & 3;
                    const int i0 = r0 + 2 * ib, c0 = j0 + 4 * cb;
                    double acc[2][4];
#pragma unroll
                    for (int r = 0; r < 2; ++r)
#pragma unroll
                        for (int q = 0; q < 4; ++q) acc[r][q] = 0.0;
                    for (int q = r0; q <= i0 + 1; ++q) {
                        const double l0 = (q <= i0) ? SE(S, i0, q) : 0.0, l1 = SE(S, i0 + 1, q);
                        double av[4];
#pragma unroll
                        for (int cc = 0; cc < 4; ++cc) av[cc] = SE(S, q, c0 + cc);
#pragma unroll
                        for (int cc = 0; cc < 4; ++cc) { acc[0][cc] = fma(l0, av[cc], acc[0][cc]); acc[1][cc] = fma(l1, av[cc], acc[1][cc]); }
                    }
#pragma unroll
                    for (int r = 0; r < 2; ++r)
#pragma unroll
                        for (int cc = 0; cc < 4; ++cc) Tb[(2 * ib + r) * 17 + 4 * cb + cc] = acc[r][cc];
                }
            }
            __syncthreads();
            // A21(i, c) = -sum_{q >= c} Tb(i, q) Dinv(q, c) ;  A11 <- Dinv
            for (int e = tid; e < R * NB; e += 256) {
                const int i = e % R, c = e / R;
                double acc = 0.0;
                for (int q = c; q < NB; ++q) acc = fma(Tb[i * 17 + q], Db[q * 17 + c], acc);
                SE(S, r0 + i, j0 + c) = -acc;
            }
            {
                const int r = tid >> 4, c = tid & 15;      // 256 threads = 16 x 16
                if (r >= c) SE(S, j0 + r, j0 + c) = Db[r * 17 + c];
            }
            __syncthreads();
        }
    }
#ifdef GPCC_PIVOT_PROF
    long long tp2 = clock64();
#endif
    // z = Linv r_k ; quad += z'z ; logdet += 2 sum log L_jj   (deterministic tree sums)
    {
        double zi = 0.0, li = 0.0;
        if (tid < BT) {
            for (int q = 0; q <= tid; ++q) zi = fma(SE(S, tid, q), rk[q], zi);
            zz[tid] = zi;
            li = log(ldiag[tid]);
        }
        double q2 = zi * zi;
        for (int o = 16; o > 0; o >>= 1) { q2 += __shfl_xor_sync(0xffffffffu, q2, o); li += __shfl_xor_sync(0xffffffffu, li, o); }
        __shared__ double redq[8], redl[8];
        if ((tid & 31) == 0) { redq[tid >> 5] = q2; redl[tid >> 5] = li; }
        __syncthreads();
        if (tid == 0) {
            double q = 0.0, ld = 0.0;
            for (int w = 0; w < 4; ++w) { q += redq[w]; ld += redl[w]; }      // threads 0..127 = warps 0..3
            a.scal[(size_t)m * 4 + 0] += 2.0 * ld;
            a.scal[(size_t)m * 4 + 1] += q;
            if (a.Tp && k == a.Tp - 1) {             // log-det and quadratic form of the shared prefix, for the other matrices
                a.scal[2] = a.scal[0];
                a.scal[3] = a.scal[1];
            }
            if (s_bad && a.info[m] == 0) a.info[m] = k * BT + s_bad;
#ifdef GPCC_PIVOT_PROF
            if (m == 0 && k == 1) printf("pivot k=1: load->chol %lld, trtri+store %lld, z/logdet %lld cycles\n", tp1 - tp0, tp2 - tp1, (long long)clock64() - tp2);
#endif
        }
    }
    if (tid < BT) a.zk[(size_t)m * BT + tid] = zz[tid];
    // Linv in panel layout: element (c, kk) = Linv[c][kk]  (coalesced: consecutive threads write consecutive doubles)
    double* gL = a.Linv + (size_t)m * TILE_ELEMS;
    for (int o = tid; o < TILE_ELEMS; o += 256) {
        const int c4 = o & 3, r8 = (o >> 2) & 7, ro = (o >> 5) & 15, k4 = o >> 9;
        gL[o] = SE(S, ro * 8 + r8, k4 * 4 + c4);
    }
    if (a.sweep) {
        if (tid < BT) {   // r_k <- Linv' z  (= D^-1 r_k)
            double s0 = 0.0;
            for (int q = tid; q < BT; ++q) s0 = fma(SE(S, q, tid), zz[q], s0);
            a.rvec[(size_t)m * a.Np + k * BT + tid] = s0;
        }
        // Dinv = Linv' Linv as an 8x8 register tile per thread (rows ty+16a, cols tx+16b) ; A_kk <- -Dinv
        double acc[8][8];
#pragma unroll
        for (int p_ = 0; p_ < 8; ++p_)
#pragma unroll
            for (int q_ = 0; q_ < 8; ++q_) acc[p_][q_] = 0.0;
        for (int q = 0; q < BT; ++q) {
            double lr[8], lc[8];
#pragma unroll
            for (int p_ = 0; p_ < 8; ++p_) { lr[p_] = SE(S, q, ty + 16 * p_); lc[p_] = SE(S, q, tx + 16 * p_); }
#pragma unroll
            for (int p_ = 0; p_ < 8; ++p_)
#pragma unroll
                for (int q_ = 0; q_ < 8; ++q_) acc[p_][q_] = fma(lr[p_], lc[q_], acc[p_][q_]);
        }
        double* gD = a.Dinv + (size_t)m * TILE_ELEMS;
#pragma unroll
        for (int p_ = 0; p_ < 8; ++p_)
#pragma unroll
            for (int q_ = 0; q_ < 8; ++q_) {
                const int r = ty + 16 * p_, c = tx + 16 * q_;
                gD[pl_off(r, c)] = acc[p_][q_];
                tile[tl_off(r, c)] = -acc[p_][q_];
            }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// gather column k of the symmetric matrix into panel layout
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gather_kernel(LargeArgs a, int k, int I0) {
    const int m = blockIdx.y;
    int I = I0 + blockIdx.x;
    if (a.sweep && I >= k) ++I;           // skip the pivot block row
    if (a.Tp && m > 0 && k < a.Tp && I < a.Tp) return;   // shared prefix rows
    if (cache_skips_row(a, k, I)) return;
    const double* mat = a.mats + (size_t)m * a.mat_stride;
    double* out = a.Pws + ((size_t)m * a.T + I) * TILE_ELEMS;
    if (I > k) {
        const double* tile = mat + tile_index(I, k) * TILE_ELEMS;
        for (int e = threadIdx.x; e < TILE_ELEMS / 2; e += 256) {      // e indexes double2 in panel layout
            const int o = e * 2;
            const int c4 = o & 3, r8 = (o >> 2) & 7, ro = (o >> 5) & 15, k4 = o >> 9;
            const int r = ro * 8 + r8, c = k4 * 4 + c4;
            *reinterpret_cast<double2*>(out + o) = *reinterpret_cast<const double2*>(tile + tl_off(r, c));
        }
    } else {
        const double* tile = mat + tile_index(k, I) * TILE_ELEMS;      // P = tile'
        for (int e = threadIdx.x; e < TILE_ELEMS; e += 256) {
            const int c4 = e & 3, r8 = (e >> 2) & 7, ro = (e >> 5) & 15, k4 = e >> 9;
            const int r = ro * 8 + r8, c = k4 * 4 + c4;
            out[e] = tile[tl_off(c, r)];
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// panel: X = P Linv' (which==0) -> panel layout (+ r_I -= X z, + forward mode write-back);  Q = P Dinv (which==1) ->
// column k of the matrix.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256, 1) panel_kernel(LargeArgs a, int k, int I0) {
    extern __shared__ __align__(128) unsigned char smraw[];
    GemmSmem& sm = *reinterpret_cast<GemmSmem*>(smraw);
    const int m = blockIdx.y, which = blockIdx.z;
    int I = I0 + blockIdx.x;
    if (a.sweep && I >= k) ++I;
    if (a.Tp && m > 0 && k < a.Tp && I < a.Tp) return;   // shared prefix rows
    if (cache_skips_row(a, k, I)) return;
    const int mL = (a.Tp && k < a.Tp) ? 0 : m;           // the pivot block of a shared step lives in matrix 0
    const double* gA = a.Pws + ((size_t)m * a.T + I) * TILE_ELEMS;
    const double* gB = (which == 0 ? a.Linv : a.Dinv) + (size_t)mL * TILE_ELEMS;
    double acc[4][8][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
    gemm_mainloop(sm, gA, gB, acc);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int ro0 = (warp & 3) * 4, co0 = (warp >> 2) * 8;
    double* mat = a.mats + (size_t)m * a.mat_stride;
    if (which == 0) {
        double* xo = a.Xws + (size_t)(k & 1) * a.x_parity_stride + ((size_t)m * a.T + I) * TILE_ELEMS;
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int mi = ro0 + i, mj = co0 + j;
                const int off = (((2 * mj + ((lane & 3) >> 1)) * 16 + mi) << 5) + ((lane >> 2) << 2) + ((lane & 1) << 1);
                *reinterpret_cast<double2*>(xo + off) = make_double2(acc[i][j][0], acc[i][j][1]);
            }
        // r_I -= X_I z_k  : partial dot over this warp's 64 columns, combined through shared memory
        double* red = reinterpret_cast<double*>(smraw);      // reuse stage memory (main loop is finished)
        __syncthreads();
        const double* z = a.zk + (size_t)mL * BT;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            double s = 0.0;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int c = (co0 + j) * 8 + (lane & 3) * 2;
                s = fma(acc[i][j][0], z[c], s);
                s = fma(acc[i][j][1], z[c + 1], s);
            }
            s += __shfl_xor_sync(0xffffffffu, s, 1);
            s += __shfl_xor_sync(0xffffffffu, s, 2);
            if ((lane & 3) == 0) red[(warp >> 2) * BT + (ro0 + i) * 8 + (lane >> 2)] = s;
        }
        __syncthreads();
        if (tid < BT) a.rvec[(size_t)m * a.Np + I * BT + tid] -= red[tid] + red[BT + tid];
        if (!a.sweep) {   // forward mode: keep L in the matrix (tile (I,k), I>k)
            double* tile = mat + tile_index(I, k) * TILE_ELEMS;
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    *reinterpret_cast<double2*>(tile + (((ro0 + i) * 16 + co0 + j) << 6) + 2 * lane) = make_double2(acc[i][j][0], acc[i][j][1]);
        }
    } else {
        if (I > k) {
            double* tile = mat + tile_index(I, k) * TILE_ELEMS;
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    *reinterpret_cast<double2*>(tile + (((ro0 + i) * 16 + co0 + j) << 6) + 2 * lane) = make_double2(acc[i][j][0], acc[i][j][1]);
        } else {       // stored transposed in tile (k, I)
            double* tile = mat + tile_index(k, I) * TILE_ELEMS;
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int r = (ro0 + i) * 8 + (lane >> 2), c = (co0 + j) * 8 + (lane & 3) * 2;
                    tile[tl_off(c, r)] = acc[i][j][0];
                    tile[tl_off(c + 1, r)] = acc[i][j][1];
                }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// update: A_IJ -= X_I X_J'  for the lower tiles not touching block k (sweep) / beyond block k (forward)
// ---------------------------------------------------------------------------------------------------------------
// phase 0: every tile; phase 1: only the tiles of block row/column k+1 (what the next pivot and panel need: the
// look-ahead part, issued on the critical stream); phase 2: all the others (issued on the bulk stream).
__device__ __forceinline__ void update_tile_of(const LargeArgs& a, int k, int phase, int tix, int& I, int& J) {
    const int n1 = k + 1;
    if (phase == 1) {
        if (a.sweep) {              // (n1, J) for J in [0, n1] \ {k}  (n1 tiles), then (I, n1) for I > n1
            if (tix < n1) { I = n1; J = tix + (tix >= k); }
            else { I = n1 + 1 + (tix - n1); J = n1; }
        } else { I = n1 + tix; J = n1; }
    } else {
        int Ir = (int)((sqrtf(8.0f * (float)tix + 1.0f) - 1.0f) * 0.5f);
        while ((size_t)Ir * (Ir + 1) / 2 > (size_t)tix) --Ir;
        while ((size_t)(Ir + 1) * (Ir + 2) / 2 <= (size_t)tix) ++Ir;
        const int Jr = tix - Ir * (Ir + 1) / 2;
        const int skip = (phase == 2) ? 2 : 1;       // blocks k (and k+1 in phase 2) are left out
        if (a.sweep) { I = Ir + (Ir >= k ? skip : 0); J = Jr + (Jr >= k ? skip : 0); }
        else { I = Ir + k + skip; J = Jr + k + skip; }
    }
}

// one 4-warp CTA per column half of a tile (GemmSmemHalf): blockIdx.x = 2 * tile + column half
__global__ void __launch_bounds__(128, 3) update_half_kernel(LargeArgs a, int k, int phase) {
    extern __shared__ __align__(128) unsigned char smraw[];
    GemmSmemHalf& sm = *reinterpret_cast<GemmSmemHalf*>(smraw);
    const int m = blockIdx.y, h = blockIdx.x & 1;
    int I, J;
    update_tile_of(a, k, phase, blockIdx.x >> 1, I, J);
    if (a.Tp && m > 0 && I < a.Tp) return;         // tile of the shared prefix (J <= I < Tp): updated once, in matrix 0
    if (cache_skips_row(a, k, J) || (a.cmode == 1 && I >= a.Tq && I < a.Tc)) return;
    const bool cached = a.cmode == 2 && k < a.Tq && I >= a.Tc;   // last band, pivot in band 1: only block (3,2) is updated,
    if (cached && J < a.Tq) return;                              // with the cached panel of the last band
    const int mB = (a.Tp && k < a.Tp && J < a.Tp) ? 0 : m;   // panel rows inside the shared prefix exist in matrix 0 only
    const double* xw = a.Xws + (size_t)(k & 1) * a.x_parity_stride;
    const double* gA = cached ? xc_tile(a, m, k, I) : xw + ((size_t)m * a.T + I) * TILE_ELEMS;
    const double* gB = xw + ((size_t)mB * a.T + J) * TILE_ELEMS;
    double* tile = a.mats + (size_t)m * a.mat_stride + tile_index(I, J) * TILE_ELEMS;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int ro0 = warp * 4, co0 = h * 8;
    double acc[4][8][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const double2 v = *reinterpret_cast<const double2*>(tile + (((ro0 + i) * 16 + co0 + j) << 6) + 2 * lane);
            acc[i][j][0] = v.x;
            acc[i][j][1] = v.y;
        }
    gemm_mainloop_half(sm, gA, gB, h, acc);
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j)
            *reinterpret_cast<double2*>(tile + (((ro0 + i) * 16 + co0 + j) << 6) + 2 * lane) = make_double2(acc[i][j][0], acc[i][j][1]);
}

// ---------------------------------------------------------------------------------------------------------------
// gradient: W = a a' - A^-1 contracted with K and dK/drho, one CTA per lower tile (one read of the inverse)
// ---------------------------------------------------------------------------------------------------------------
template <int KID>
__global__ void __launch_bounds__(256) gradreduce_kernel(EvalBatch b, int e0, LargeArgs a) {
    __shared__ double tr[BT], tc[BT], ar[BT], ac[BT], wr[BT], wc[BT];
    __shared__ double rows[1][BT], cols[8][BT];
    __shared__ double esum[8];
    const int m = blockIdx.y, e = e0 + m;
    const int tix = blockIdx.x;
    int I = (int)((sqrtf(8.0f * (float)tix + 1.0f) - 1.0f) * 0.5f);
    while ((size_t)I * (I + 1) / 2 > (size_t)tix) --I;
    while ((size_t)(I + 1) * (I + 2) / 2 <= (size_t)tix) ++I;
    const int J = tix - I * (I + 1) / 2;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid < BT) {
        const int i = I * BT + tid;
        tr[tid] = a.tsh[(size_t)m * a.Np + i]; ar[tid] = a.av[(size_t)m * a.Np + i]; wr[tid] = i < a.N ? a.rvec[(size_t)m * a.Np + i] : 0.0;
    } else {
        const int c = tid - BT, j = J * BT + c;
        tc[c] = a.tsh[(size_t)m * a.Np + j]; ac[c] = a.av[(size_t)m * a.Np + j]; wc[c] = j < a.N ? a.rvec[(size_t)m * a.Np + j] : 0.0;
    }
    for (int q = tid; q < 8 * BT; q += 256) (&cols[0][0])[q] = 0.0;
    if (tid < BT) rows[0][tid] = 0.0;
    __syncthreads();
    const KernParams kp = make_kern_params(KID, b.rho[e]);
    const double* tile = a.mats + (size_t)m * a.mat_stride + tile_index(I, J) * TILE_ELEMS;
    const int rr = lane >> 2, cc = (lane & 3) * 2;
    double es = 0.0;
    // warp w handles micro-tile rows mi = 2w, 2w+1 (all 16 mj): row sums stay in the warp, column sums go to cols[w][]
    for (int mi = 2 * warp; mi < 2 * warp + 2; ++mi) {
        const int r = mi * 8 + rr;
        double rsum = 0.0;
        for (int mj = 0; mj < 16; ++mj) {
            const double2 v = *reinterpret_cast<const double2*>(tile + ((mi * 16 + mj) << 6) + 2 * lane);
            const double vv[2] = {v.x, v.y};
            double csum[2];
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const int c = mj * 8 + cc + q;
                const int gi = I * BT + r, gj = J * BT + c;
                const double W = fma(wr[r], wc[c], vv[q]);              // a_i a_j - (A^-1)_ij   (matrix holds -A^-1)
                double kv, dkv;
                kern_value_drho<KID>(tr[r] - tc[c], kp, kv, dkv);
                const double aa = ar[r] * ac[c];
                double ct = W * (aa * kv), et = W * (aa * dkv);
                if (I == J) {
                    if (gi == gj) { rsum += ct; ct = 0.0; et = 0.0; }
                    else if (gj > gi) { ct = 0.0; et = 0.0; }
                }
                rsum += ct;
                csum[q] = ct;
                es += et;
            }
            // column sums over the 8 rows of this micro tile: lanes with equal (lane&3) hold the same columns
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                double s = csum[q];
                s += __shfl_xor_sync(0xffffffffu, s, 4);
                s += __shfl_xor_sync(0xffffffffu, s, 8);
                s += __shfl_xor_sync(0xffffffffu, s, 16);
                if (rr == 0) cols[warp][mj * 8 + cc + q] += s;
            }
        }
        rsum += __shfl_xor_sync(0xffffffffu, rsum, 1);
        rsum += __shfl_xor_sync(0xffffffffu, rsum, 2);
        if ((lane & 3) == 0) rows[0][r] = rsum;
    }
    for (int o = 16; o > 0; o >>= 1) es += __shfl_xor_sync(0xffffffffu, es, o);
    if (lane == 0) esum[warp] = es;
    __syncthreads();
    double* part = a.part + (size_t)m * a.T * a.T * BT;
    if (tid < BT) {
        double cs = 0.0;
        for (int w = 0; w < 8; ++w) cs += cols[w][tid];
        if (I == J) {
            part[((size_t)I * a.T + J) * BT + tid] = rows[0][tid] + cs;
        } else {
            part[((size_t)I * a.T + J) * BT + tid] = rows[0][tid];
            part[((size_t)J * a.T + I) * BT + tid] = cs;
        }
    }
    if (tid == 0) {
        double s = 0.0;
        for (int w = 0; w < 8; ++w) s += esum[w];
        a.epart[(size_t)m * (a.T * (a.T + 1) / 2) + tix] = s;
    }
}

__global__ void __launch_bounds__(256) finalize_kernel(DevProblem p, EvalBatch b, int e0, LargeArgs a) {
    __shared__ double red[8];
    __shared__ double srow_band[MAX_BANDS];
    const int m = blockIdx.x, e = e0 + m, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int info = a.info[m];
    double logdet = a.scal[(size_t)m * 4 + 0], quad = a.scal[(size_t)m * 4 + 1];
    if (a.Tp && m > 0) {                          // add the shared prefix (computed in matrix 0)
        logdet += a.scal[2];
        quad += a.scal[3];
        const int i0 = a.info[0];
        if (i0 != 0 && i0 <= a.Tp * BT) info = i0; // the first failing leading minor lies inside the prefix
    }
    const double ll = -0.5 * ((double)a.N * LOG2PI + logdet + quad);
    if (tid == 0) {
        b.ll[e] = info ? -INFINITY : ll;
        if (b.info) b.info[e] = info;
    }
    if (!b.want_grad) return;
    if (info) { if (tid <= a.L) b.grad[(size_t)e * (a.L + 1) + tid] = 0.0; return; }
    const double* part = a.part + (size_t)m * a.T * a.T * BT;
    for (int pb = 0; pb < a.L; ++pb) {
        double s = 0.0;
        for (int i = p.band_start[pb] + tid; i < p.band_start[pb + 1]; i += 256) {
            const int I = i >> 7, r = i & 127;
            double si = 0.0;
            for (int src = 0; src < a.T; ++src) si += part[((size_t)I * a.T + src) * BT + r];
            s += si;
        }
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        __syncthreads();
        if (lane == 0) red[warp] = s;
        __syncthreads();
        if (tid == 0) {
            double v = 0.0;
            for (int w = 0; w < 8; ++w) v += red[w];
            srow_band[pb] = v;
        }
    }
    double es = 0.0;
    const int nt = a.T * (a.T + 1) / 2;
    for (int q = tid; q < nt; q += 256) es += a.epart[(size_t)m * nt + q];
    for (int o = 16; o > 0; o >>= 1) es += __shfl_xor_sync(0xffffffffu, es, o);
    __syncthreads();
    if (lane == 0) red[warp] = es;
    __syncthreads();
    if (tid == 0) {
        double v = 0.0;
        for (int w = 0; w < 8; ++w) v += red[w];
        for (int pb = 0; pb < a.L; ++pb) b.grad[(size_t)e * (a.L + 1) + pb] = srow_band[pb] / b.alpha[(size_t)e * a.L + pb];
        b.grad[(size_t)e * (a.L + 1) + a.L] = v;
    }
}

// last-band cache, FILL side: the panels of step k (rows of the last band) ...
__global__ void __launch_bounds__(256) export_x_kernel(LargeArgs a, int k) {
    const int m = blockIdx.y, I = a.Tc + blockIdx.x;
    const double2* src = reinterpret_cast<const double2*>(a.Xws + (size_t)(k & 1) * a.x_parity_stride + ((size_t)m * a.T + I) * TILE_ELEMS);
    double2* dst = reinterpret_cast<double2*>(xc_tile(a, m, k, I));
    for (int q = threadIdx.x; q < TILE_ELEMS / 2; q += 256) dst[q] = src[q];
}
// ... and, after step Tq-1, the state of block (3,3) (blockIdx.x < number of its tiles) and of r_3 (the last block)
__global__ void __launch_bounds__(256) export_state_kernel(LargeArgs a) {
    const int m = blockIdx.y, nC = a.T - a.Tc, ntc = nC * (nC + 1) / 2;
    if ((int)blockIdx.x == ntc) {
        double* dst = a.RC + (size_t)a.slot[m] * a.rc_stride;
        const double* src = a.rvec + (size_t)m * a.Np + (size_t)a.Tc * BT;
        for (int q = threadIdx.x; q < nC * BT; q += 256) dst[q] = src[q];
        return;
    }
    const int tix = blockIdx.x;
    int I = (int)((sqrtf(8.0f * (float)tix + 1.0f) - 1.0f) * 0.5f);
    while (I * (I + 1) / 2 > tix) --I;
    while ((I + 1) * (I + 2) / 2 <= tix) ++I;
    const int J = tix - I * (I + 1) / 2;
    const double2* src = reinterpret_cast<const double2*>(a.mats + (size_t)m * a.mat_stride + tile_index(I + a.Tc, J + a.Tc) * TILE_ELEMS);
    double2* dst = reinterpret_cast<double2*>(ac_tile(a, m, I + a.Tc, J + a.Tc));
    for (int q = threadIdx.x; q < TILE_ELEMS / 2; q += 256) dst[q] = src[q];
}

// dense column-major Cholesky factor (lower triangle, zeros above) out of the tile layout: forward mode only
__global__ void dump_chol_kernel(EvalBatch b, int e0, LargeArgs a) {
    const int m = blockIdx.y, e = e0 + m;
    const double* mat = a.mats + (size_t)m * a.mat_stride;
    double* out = b.dump_chol + (size_t)e * a.N * a.N;
    const size_t total = (size_t)a.N * a.N;
    for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < total; q += (size_t)gridDim.x * blockDim.x) {
        const int i = (int)(q % a.N), j = (int)(q / a.N);
        out[q] = i >= j ? mat[tile_index(i >> 7, j >> 7) * TILE_ELEMS + tl_off(i & 127, j & 127)] : 0.0;
    }
}

}  // namespace

// Last-band cache: [slots][...] per array.
struct TauCache {
    DevArray<double> XC, AC, RC;
    int slots = 0, Tc = 0, Tq = 0;
    size_t xc_stride = 0, ac_stride = 0, rc_stride = 0;   // doubles per slot
};

// Workspace of one shape: N, and B matrices per wave.  ensure() builds a new one whenever N changes or B must grow.
struct LargeImpl {
    int dev = 0;
    int N = 0, T = 0, Np = 0, B = 0;
    size_t mat_stride = 0;
    DevArray<double> mats, Pws, Xws, Linv, Dinv, rvec, zk, scal, tsh, av, part, epart;
    DevArray<int> info;
    DevArray<int> eidx_d, slot_d;                // [B] per-wave maps of the last-band cache
    std::unique_ptr<TauCache> cache;
    Event ev[4];
    Stream bulk;                                 // second stream: the bulk of each trailing update (look-ahead)
    Event ev_panel[2], ev_bulk[2];
    bool attr_set = false;
    ~LargeImpl() { cudaSetDevice(dev); }
};

void LargeImplDelete::operator()(LargeImpl* w) const { delete w; }

namespace {

// The old workspace is freed before the new one is allocated, so that peak memory is one workspace.  On failure `ws` is
// empty and the next call allocates again.
cudaError_t ensure(LargeWorkspace& ws, int N, int want_B) {
    const int T = (N + BT - 1) / BT;
    if (ws && ws->N == N && ws->B >= want_B) return cudaSuccess;
    ws.reset();
    LargeWorkspace w(new LargeImpl());
    cudaError_t e = cudaGetDevice(&w->dev);
    if (e != cudaSuccess) return e;
    const int Np = T * BT;
    const size_t ntiles = (size_t)T * (T + 1) / 2;
    const size_t mat_stride = ntiles * TILE_ELEMS;
    size_t free_b = 0, total_b = 0;
    e = cudaMemGetInfo(&free_b, &total_b);
    if (e != cudaSuccess) return e;
    const size_t per = (mat_stride + 3 * (size_t)T * TILE_ELEMS + 2 * TILE_ELEMS + (size_t)T * T * BT + ntiles + 4 * (size_t)Np) * sizeof(double);
    int B = want_B;
    while (B > 1 && (size_t)B * per > free_b / 2) B /= 2;
    if ((size_t)B * per > free_b) return cudaErrorMemoryAllocation;
#define ALLOC(arr, n) if ((e = w->arr.reserve((size_t)(n))) != cudaSuccess) return e;
    ALLOC(mats, (size_t)B * mat_stride)
    ALLOC(Pws, (size_t)B * T * TILE_ELEMS)
    ALLOC(Xws, (size_t)2 * B * T * TILE_ELEMS)
    ALLOC(Linv, (size_t)B * TILE_ELEMS)
    ALLOC(Dinv, (size_t)B * TILE_ELEMS)
    ALLOC(rvec, (size_t)B * Np)
    ALLOC(zk, (size_t)B * BT)
    ALLOC(scal, (size_t)B * 4)
    ALLOC(tsh, (size_t)B * Np)
    ALLOC(av, (size_t)B * Np)
    ALLOC(part, (size_t)B * T * T * BT)
    ALLOC(epart, (size_t)B * ntiles)
    ALLOC(info, (size_t)B)
    ALLOC(eidx_d, (size_t)B)
    ALLOC(slot_d, (size_t)B)
#undef ALLOC
    for (auto& ev : w->ev) if ((e = create_event(ev)) != cudaSuccess) return e;
    for (auto& ev : w->ev_panel) if ((e = create_event(ev, cudaEventDisableTiming)) != cudaSuccess) return e;
    for (auto& ev : w->ev_bulk) if ((e = create_event(ev, cudaEventDisableTiming)) != cudaSuccess) return e;
    int prio_lo = 0, prio_hi = 0;
    if ((e = cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi)) != cudaSuccess) return e;
    if ((e = create_stream(w->bulk, prio_lo)) != cudaSuccess) return e;
    w->N = N; w->T = T; w->Np = Np; w->B = B; w->mat_stride = mat_stride;
    ws = std::move(w);
    return cudaSuccess;
}

// Last-band cache: room for `slots` distinct values of the last delay.  Returns false (no error) when it does not fit; the
// cache is then empty.
bool ensure_cache(LargeImpl& w, int slots, int Tq, int Tc) {
    const TauCache* old = w.cache.get();
    if (old && old->slots >= slots && old->Tc == Tc && old->Tq == Tq) return true;
    w.cache.reset();
    auto c = std::make_unique<TauCache>();
    const int nC = w.T - Tc;
    const int wanted = slots;
    c->xc_stride = (size_t)Tq * nC * TILE_ELEMS;
    c->ac_stride = (size_t)nC * (nC + 1) / 2 * TILE_ELEMS;
    c->rc_stride = (size_t)nC * BT;
    const size_t bytes = (size_t)slots * (c->xc_stride + c->ac_stride + c->rc_stride) * sizeof(double);
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess || bytes > free_b / 2) return false;
    // head-room (a grid has ~10^2 distinct delays per band): a first call with a few candidates must not force a re-allocation,
    // and its allocator stall, into the next one
    while (slots < 128 && (size_t)(2 * slots) * (bytes / wanted) <= free_b / 8) slots *= 2;
    if (c->XC.reserve((size_t)slots * c->xc_stride) != cudaSuccess || c->AC.reserve((size_t)slots * c->ac_stride) != cudaSuccess ||
        c->RC.reserve((size_t)slots * c->rc_stride) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    c->slots = slots; c->Tc = Tc; c->Tq = Tq;
    w.cache = std::move(c);
    return true;
}

// cmode 0: plain wave.  1: FILL wave of the last-band cache (matrix m = evaluation h_eidx[m], result into slot h_slot[m]; only the
// steps k < Tq run, nothing is reported).  2: USE wave (matrix m reads slot h_slot[m]).
template <int KID>
cudaError_t run_wave(const DevProblem& p, const EvalBatch& b, int e0, int nb, int Tp, LargeImpl& w, cudaStream_t st, bool profile,
                     LargeTimings* tm, int cmode = 0, int Tq = 0, int Tc = 0, const int* h_eidx = nullptr, const int* h_slot = nullptr) {
    LargeArgs a{};
    a.N = p.N; a.L = p.L; a.T = w.T; a.Np = w.Np; a.kid = KID;
    a.sweep = b.want_grad ? 1 : 0;
    a.Tp = a.sweep ? 0 : Tp;
    a.mode_postb = b.mode_postb;
    a.mats = w.mats.d; a.Pws = w.Pws.d; a.Xws = w.Xws.d; a.Linv = w.Linv.d; a.Dinv = w.Dinv.d; a.rvec = w.rvec.d; a.zk = w.zk.d;
    a.scal = w.scal.d; a.info = w.info.d; a.tsh = w.tsh.d; a.av = w.av.d; a.part = w.part.d; a.epart = w.epart.d; a.mat_stride = w.mat_stride;
    a.x_parity_stride = (size_t)w.B * w.T * TILE_ELEMS;
    a.cmode = a.sweep ? 0 : cmode; a.Tq = Tq; a.Tc = Tc;
    a.eidx = nullptr; a.slot = w.slot_d.d;
    if (const TauCache* c = w.cache.get()) {
        a.XC = c->XC.d; a.AC = c->AC.d; a.RC = c->RC.d; a.xc_stride = c->xc_stride; a.ac_stride = c->ac_stride; a.rc_stride = c->rc_stride;
    }
    if (a.cmode) {      // pageable source: the copy is staged before the call returns; ordered behind the previous wave on `st`
        cudaMemcpyAsync(w.slot_d.d, h_slot, (size_t)nb * sizeof(int), cudaMemcpyHostToDevice, st);
        if (a.cmode == 1) {
            cudaMemcpyAsync(w.eidx_d.d, h_eidx, (size_t)nb * sizeof(int), cudaMemcpyHostToDevice, st);
            a.eidx = w.eidx_d.d;
            a.Tp = Tq;      // the matrices of a FILL wave share band 1 (same hyper-parameters, same first delay)
        }
    }
    const int T = w.T;
    const int ksteps = a.cmode == 1 ? Tq : T;
    const int ntiles = T * (T + 1) / 2;
    const size_t gemm_smem = sizeof(GemmSmem) + 128;
    const size_t pivot_smem = (size_t)(BT * PLD + 3 * BT + 112 * 17 + 16 * 17) * sizeof(double);
    if (!w.attr_set) {
        cudaFuncSetAttribute(panel_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gemm_smem);
        cudaFuncSetAttribute(update_half_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(GemmSmemHalf) + 128));
        cudaFuncSetAttribute(pivot_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pivot_smem);
        w.attr_set = true;
    }
    const size_t half_smem = sizeof(GemmSmemHalf) + 128;
    auto launch_update = [&](int ntile, int phase, int kk, cudaStream_t strm) {
        update_half_kernel<<<dim3(2 * ntile, nb), 128, half_smem, strm>>>(a, kk, phase);
    };
    long long launches = 0;
    if (profile) cudaEventRecord(w.ev[0].get(), st);
    prep_kernel<<<dim3((w.Np + 255) / 256, nb), 256, 0, st>>>(p, b, e0, a);
    assemble_kernel<KID><<<dim3(ntiles, nb), 256, 0, st>>>(p, b, e0, a);
    launches += 2;
    {   // HBM bytes the assembly of this wave moves (what the kernel's early exits leave): tiles written, imported tiles read + written
        auto tri = [](long long n) { return n * (n + 1) / 2; };
        const long long nC = T - Tc, nM = Tc - Tq;
        long long own = ntiles, lead = 0;                    // tiles per matrix, extra tiles of matrix 0 (the shared prefix)
        if (a.Tp) { lead = tri(a.Tp); own = ntiles - lead; }
        if (a.cmode == 1) own = nC * Tq + tri(nC);           // FILL: blocks (3,1) and (3,3)
        if (a.cmode == 2) own += tri(nC) - nC * Tq;          // USE: block (3,1) not assembled, block (3,3) read + written
        tm->assembly_bytes += ((long long)nb * own + lead) * (long long)(TILE_ELEMS * sizeof(double));
        (void)nM;
    }
    if (profile) cudaEventRecord(w.ev[1].get(), st);
    // Look-ahead schedule on two streams.  Critical stream `st`: pivot_k, gather_k, panel_k, then the part of update k
    // that touches block row/column k+1, so that pivot/gather/panel of step k+1 start while the bulk stream is still
    // busy with the rest of update k (the pivot kernel occupies one SM per matrix; without look-ahead the other SMs idle).
    static const bool lookahead = !(getenv("GPCC_LARGE_NO_LOOKAHEAD"));
    bool bulk_pending[2] = {false, false};
    for (int k = 0; k < ksteps; ++k) {
        pivot_kernel<<<nb, 256, pivot_smem, st>>>(a, k);
        ++launches;
        const int I0 = a.sweep ? 0 : k + 1;
        const int nI = a.sweep ? T - 1 : T - 1 - k;
        if (nI <= 0) continue;
        gather_kernel<<<dim3(nI, nb), 256, 0, st>>>(a, k, I0);
        panel_kernel<<<dim3(nI, nb, a.sweep ? 2 : 1), 256, gemm_smem, st>>>(a, k, I0);
        launches += 2;
        if (a.cmode == 1) { export_x_kernel<<<dim3(T - Tc, nb), 256, 0, st>>>(a, k); ++launches; }
        const bool has_next = (k + 1 < T);
        const int n_crit = a.sweep ? T - 1 : T - 1 - k;                 // tiles of block row/column k+1
        const int n_rest_side = a.sweep ? T - 2 : T - 2 - k;
        const int n_rest = n_rest_side > 0 ? n_rest_side * (n_rest_side + 1) / 2 : 0;
        if (!lookahead || !has_next) {
            if (bulk_pending[(k + 1) & 1]) { cudaStreamWaitEvent(st, w.ev_bulk[(k + 1) & 1].get(), 0); bulk_pending[(k + 1) & 1] = false; }
            launch_update(nI * (nI + 1) / 2, 0, k, st);
            ++launches;
            continue;
        }
        cudaEventRecord(w.ev_panel[k & 1].get(), st);
        // the critical tiles were last written by the bulk part of update k-1
        if (bulk_pending[(k + 1) & 1]) { cudaStreamWaitEvent(st, w.ev_bulk[(k + 1) & 1].get(), 0); bulk_pending[(k + 1) & 1] = false; }
        launch_update(n_crit, 1, k, st);
        ++launches;
        if (n_rest > 0) {
            cudaStreamWaitEvent(w.bulk.get(), w.ev_panel[k & 1].get(), 0);
            launch_update(n_rest, 2, k, w.bulk.get());
            cudaEventRecord(w.ev_bulk[k & 1].get(), w.bulk.get());
            bulk_pending[k & 1] = true;
            ++launches;
        }
    }
    for (int q = 0; q < 2; ++q)
        if (bulk_pending[q]) cudaStreamWaitEvent(st, w.ev_bulk[q].get(), 0);
    if (profile) cudaEventRecord(w.ev[2].get(), st);
    if (a.cmode == 1) {
        const int nC = T - Tc;
        export_state_kernel<<<dim3(nC * (nC + 1) / 2 + 1, nb), 256, 0, st>>>(a);
        ++launches;
    }
    if (b.want_grad) {
        gradreduce_kernel<KID><<<dim3(ntiles, nb), 256, 0, st>>>(b, e0, a);
        ++launches;
    }
    if (a.cmode != 1) { finalize_kernel<<<nb, 256, 0, st>>>(p, b, e0, a); ++launches; }
    if (b.dump_chol && !a.sweep) {
        dump_chol_kernel<<<dim3(592, nb), 256, 0, st>>>(b, e0, a);
        ++launches;
    }
    if (profile) cudaEventRecord(w.ev[3].get(), st);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    if (profile) {
        e = cudaEventSynchronize(w.ev[3].get());
        if (e != cudaSuccess) return e;
        float t01 = 0, t12 = 0, t23 = 0;
        cudaEventElapsedTime(&t01, w.ev[0].get(), w.ev[1].get());
        cudaEventElapsedTime(&t12, w.ev[1].get(), w.ev[2].get());
        cudaEventElapsedTime(&t23, w.ev[2].get(), w.ev[3].get());
        tm->ms_assembly += t01; tm->ms_factor += t12; tm->ms_gradreduce += t23;
    }
    tm->launches += launches;
    return cudaSuccess;
}

}  // namespace

cudaError_t large_eval(const DevProblem& p, const EvalBatch& b, LargeWorkspace& ws, cudaStream_t stream, bool profile,
                       LargeTimings* tm) {
    // Matrices per wave.  The pivot kernel is one CTA per matrix and its 128-column chain is the critical path of a block step;
    // a wave must hold enough matrices for the DMMA trailing updates of the others to cover it (measured at N = 6144: 8 per
    // wave 21.6 TFLOP/s, pivot bound; 32 per wave update bound).  ensure() halves the wave if memory is short.
    static const int wave_env = getenv("GPCC_LARGE_WAVE") ? atoi(getenv("GPCC_LARGE_WAVE")) : 0;
    const int want_B = std::min(b.M, wave_env > 0 ? wave_env : (p.N >= 8192 ? 16 : (p.N >= 4096 ? 32 : (p.N >= 1024 ? 128 : 512))));
    cudaError_t e = ensure(ws, p.N, std::max(want_B, 1));
    if (e != cudaSuccess) return e;
    LargeImpl& w = *ws;
    // Structure reuse across the grid (SURVEY.md 8f item 2; src/delayedCovariance.jl:23-31: block (l, m) of the covariance depends
    // on tau_l - tau_m only).  Evaluations that share the hyper-parameters and the delays of all bands but the last have an
    // identical leading principal block; in forward (Cholesky) mode a wave made of such a run factorises that block ONCE.
    // The callers sort fixed-theta sweeps so that these runs are long (api.cu); here consecutive runs are detected on the host
    // mirrors of the parameters and cut into balanced waves.
    static const bool no_share = getenv("GPCC_LARGE_NO_SHARE") != nullptr;
    const int L = p.L;
    const int Tp_full = (L >= 2 && !b.want_grad && !no_share && b.h_delays && b.h_alpha && b.h_rho) ? p.band_start[L - 1] / BT : 0;
    auto same_prefix = [&](int x, int y) {
        if (b.h_rho[x] != b.h_rho[y]) return false;
        for (int l = 0; l < L; ++l) if (b.h_alpha[(size_t)x * L + l] != b.h_alpha[(size_t)y * L + l]) return false;
        for (int l = 0; l + 1 < L; ++l) if (b.h_delays[(size_t)x * L + l] != b.h_delays[(size_t)y * L + l]) return false;
        return true;
    };
    long long shared_evals = 0;
    std::vector<int> rl;                                     // rl[x] = length of the run with a common prefix that starts at x
    if (Tp_full > 0) {
        rl.assign(b.M, 1);
        for (int x = b.M - 2; x >= 0; --x) if (same_prefix(x, x + 1)) rl[x] = rl[x + 1] + 1;
    }
    // Last-band cache (three or more bands, one theta and one first delay for the whole batch -- the fixed-theta grid sweep): what
    // the band-1 steps do to the rows of the last band depends on the last delay alone (written for three bands below).  A grid has far fewer
    // distinct tau_3 than candidates, so those steps run once per distinct value (FILL waves) and every candidate imports
    // their result (USE): per candidate 4.3 n^3 + the amortised fill instead of 6.3 n^3 flop (n = points per band), bitwise the
    // same tiles as without the cache (same kernels, same operands, same order).
    static const bool no_cache = getenv("GPCC_LARGE_NO_TAUCACHE") != nullptr;
    bool use_cache = false;
    int Tq = 0, Tc = 0, nslots = 0;
    std::vector<int> slot_of, rep;
    if (Tp_full > 0 && L >= 3 && !no_cache && !b.dump_chol && !b.mode_postb && p.band_start[1] >= BT && b.M >= 8) {
        bool same = true;
        for (int x = 1; x < b.M && same; ++x) {
            same = memcmp(&b.h_rho[x], &b.h_rho[0], sizeof(double)) == 0 &&
                   memcmp(&b.h_alpha[(size_t)x * L], &b.h_alpha[0], L * sizeof(double)) == 0 &&
                   memcmp(&b.h_delays[(size_t)x * L], &b.h_delays[0], sizeof(double)) == 0;
        }
        if (same) {
            std::map<uint64_t, int> ids;
            slot_of.resize(b.M);
            for (int x = 0; x < b.M; ++x) {
                uint64_t bits;
                memcpy(&bits, &b.h_delays[(size_t)x * L + L - 1], sizeof(bits));
                auto it = ids.find(bits);
                if (it == ids.end()) { it = ids.emplace(bits, (int)rep.size()).first; rep.push_back(x); }
                slot_of[x] = it->second;
            }
            nslots = (int)rep.size();
            Tq = p.band_start[1] / BT;                   // block columns entirely inside band 1
            Tc = (p.band_start[L - 1] + BT - 1) / BT;    // block rows entirely inside the last band (a row of tiles that straddles
                                                         // its boundary is handled like the middle bands: per candidate)
            // worth it when a slot serves several candidates (the fill of a slot costs about a third of a candidate)
            if (b.M >= 3 * nslots && Tc < w.T && ensure_cache(w, nslots, Tq, Tc)) use_cache = true;
        }
    }
    auto dispatch = [&](int e0, int nb, int Tp, int cmode, const int* h_eidx, const int* h_slot) {
        switch (p.kernel_id) {
            case K_OU:  return run_wave<K_OU>(p, b, e0, nb, Tp, w, stream, profile, tm, cmode, Tq, Tc, h_eidx, h_slot);
            case K_RBF: return run_wave<K_RBF>(p, b, e0, nb, Tp, w, stream, profile, tm, cmode, Tq, Tc, h_eidx, h_slot);
            case K_M32: return run_wave<K_M32>(p, b, e0, nb, Tp, w, stream, profile, tm, cmode, Tq, Tc, h_eidx, h_slot);
            default:    return run_wave<K_M52>(p, b, e0, nb, Tp, w, stream, profile, tm, cmode, Tq, Tc, h_eidx, h_slot);
        }
    };
    if (use_cache) {
        std::vector<int> ids(w.B);
        for (int s0 = 0; s0 < nslots; s0 += w.B) {
            const int nb = std::min(w.B, nslots - s0);
            for (int m = 0; m < nb; ++m) ids[m] = s0 + m;
            e = dispatch(0, nb, 0, 1, rep.data() + s0, ids.data());
            if (e != cudaSuccess) return e;
        }
        tm->tau_cache_evals += b.M;
    }
    constexpr int MIN_RUN = 4;
    for (int e0 = 0; e0 < b.M;) {
        int nb = 0, Tp = 0;
        if (Tp_full > 0 && rl[e0] >= MIN_RUN) {              // balanced waves inside the run
            const int nwaves = (rl[e0] + w.B - 1) / w.B;
            nb = (rl[e0] + nwaves - 1) / nwaves;
            Tp = Tp_full;
            shared_evals += nb - 1;
        } else {                                             // no sharing: up to a full wave, but stop where a long run begins
            while (nb < w.B && e0 + nb < b.M && !(nb > 0 && Tp_full > 0 && rl[e0 + nb] >= MIN_RUN)) ++nb;
        }
        e = dispatch(e0, nb, Tp, use_cache ? 2 : 0, nullptr, use_cache ? slot_of.data() + e0 : nullptr);
        if (e != cudaSuccess) return e;
        e0 += nb;
    }
    tm->shared_prefix_evals += shared_evals;
    return cudaSuccess;
}

}  // namespace gpcc
