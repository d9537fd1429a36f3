// Fused small-N evaluator, the device function shared by the batch kernel (small_sweep.cu: one CTA per (delay candidate,
// hyper-parameter) pair) and by the device-resident fit (small_fit.cu: one persistent CTA per candidate).
//
// Replaces, for N+1 <= 8*SMALL_MAX_T, the reference's objective
//   K = delayedCovariance(kernel, alpha, tau, rho, tarray) + Sobs + B ; logpdf(MvNormal(bbar, K), Y)
// (/root/reference/src/gpccfixdelay_marginaliseb.jl:133-141, src/delayedCovariance.jl:1-38) and adds
// the analytic gradient 0.5 tr((a a' - K^-1) dK/dtheta) that north_star asks for.
//
// Design (B200: 64 FP64 FMA/clk/SM, 64K registers/SM, smem 128 B/clk):
//   * the lower triangle of the (N+1)x(N+1) bordered matrix [K~ r; r' 0] lives ENTIRELY IN REGISTERS,
//     one 8x8 tile per thread (N=150 -> 190 threads x 64 doubles); nothing N^2-sized touches smem/HBM;
//   * assembly is fused: every thread evaluates its 64 kernel entries from the shifted times in smem;
//   * one symmetric Gauss-Jordan "sweep" per index k (k = 0..N-1): A_ij -= A_ik A_kj / A_kk for
//     i,j != k, A_ik <- A_ik/A_kk, A_kk <- -1/A_kk.  Per step a thread does 64 independent DFMAs on its
//     tile from 16 values broadcast through shared memory (16 LDS.64) and ONE __syncthreads: the
//     owners publish column k+1 (double buffered) as soon as their slice of it is updated.
//     The pivots are exactly the Cholesky pivots L_kk^2, so logdet = sum log(pivot) and the
//     leading-minor `info` follow LAPACK dpotrf; the border row gives a = K~^-1 r and the corner
//     -r'K~^-1 r by forward elimination; after N steps the tile registers hold -K~^-1.
//     Work: N^3/2 DFMA = N^3 flop, the same as potrf + potri, but perfectly balanced, with no
//     triangular solves and no second pass;
//   * forward-only mode (no gradient wanted): plain Gaussian elimination.  Only the tiles with tj >= tk still change
//     something that is read later (the pivots and the border row); the others skip the step, so the work is N^3/3 flop.
//     The elements that feed the pivots and the corner see exactly the operations of the full sweep: logL is bitwise the
//     same.  Tiles are then dealt to threads column by column, so that the tiles which have left the elimination are a
//     prefix of the thread range and whole warps retire as the pivot moves on;
//   * the gradient contracts W = a a' - K~^-1 against K and dK/drho recomputed on the fly (never
//     stored), reduced deterministically (no atomics).
#pragma once
#include "gpcc_internal.h"
#include "kernfun.cuh"
#include <climits>
#include <cmath>
#include <type_traits>

namespace gpcc {
namespace small {

#ifdef GPCC_STEP_PROF
__device__ unsigned* gpcc_prof_out;
__device__ int gpcc_prof_block;
#endif

constexpr int TS = SMALL_TILE;  // 8
constexpr double LOG2PI = 1.8378770664093454835606594728112;

// Chunked layout of the per-point vectors in shared memory: [in-tile index (8)][tile (<=32)], with a compile-time part
// stride so that every address in the sweep loop is "per-thread base + immediate".  No two values that one thread reads
// are adjacent, so every access is a 64-bit LDS/STS: a 128-bit access needs an aligned quad of destination registers,
// which ptxas cannot find among the 128 accumulator registers of the tile, and it lands the quad in scratch registers
// and copies the values out (14-59 moves per sweep step with the former [pair of rows][tile][2] layout).
constexpr int CS = 32;          // doubles per part (>= SMALL_MAX_T)
constexpr int VLEN = 8 * CS;    // doubles per vector
__device__ __forceinline__ int cidx(int i) { return (i & 7) * CS + (i >> 3); }
__device__ __forceinline__ void load8(const double* buf, int tile, double (&out)[8]) {
#pragma unroll
    for (int r = 0; r < 8; ++r) out[r] = buf[r * CS + tile];
}
__device__ __forceinline__ void store8(double* buf, int tile, const double (&in)[8]) {
#pragma unroll
    for (int r = 0; r < 8; ++r) buf[r * CS + tile] = in[r];
}

// shared-memory footprint of one evaluation (doubles, then Np ints)
__host__ __device__ inline size_t eval_smem_bytes(int T, int want_grad) {
    const int Np = T * TS;
    const size_t doubles = (size_t)VLEN * 10 + 4 + 64 + (want_grad ? (size_t)T * T * 8 : 0);
    return doubles * sizeof(double) + (size_t)Np * sizeof(int) + 16;
}

// Occupancy instantiation <MAXTHREADS, MINBLOCKS> of the batch kernel (small_sweep.cu) and of the fit kernel (small_fit.cu)
// by tile count T, batch size M and the SM count of the device (measured on B200, profiles/small_sweep_variants_r1.log):
//   N <= 119 (T <= 15: 120 tiles, 128 threads): three CTAs per SM are 8 % faster once every SM has three (32.7 vs
//   35.6 us per evaluation and SM), but slower when the batch leaves SMs with one or two (82 vs 65 us at one CTA per SM);
//   N <= 151 (192 threads): a CTA that is alone on its SM runs faster with 255 registers and no spills (101 vs 122 us),
//   two co-resident CTAs at 168 registers win as soon as there is more than one evaluation per SM (134 vs 188 us for two).
// Returns f(std::integral_constant<int, MAXTHREADS>, std::integral_constant<int, MINBLOCKS>, threads, maxT): threads is the
// block size for T (its tiles in whole warps), maxT the largest T the instantiation serves.
template <class F>
cudaError_t with_instantiation(int T, int M, int nsm, F&& f) {
    using std::integral_constant;
    const int threads = (T * (T + 1) / 2 + 31) / 32 * 32;
    if (threads <= 128) {
        if (M >= 3 * nsm) return f(integral_constant<int, 128>(), integral_constant<int, 3>(), threads, 15);
        return f(integral_constant<int, 128>(), integral_constant<int, 2>(), threads, 15);
    }
    if (threads <= 192 && M > nsm) return f(integral_constant<int, 192>(), integral_constant<int, 2>(), threads, 19);
    if (threads <= 224) return f(integral_constant<int, 224>(), integral_constant<int, 1>(), threads, 20);
    return f(integral_constant<int, 352>(), integral_constant<int, 1>(), threads, SMALL_MAX_T);
}

#ifdef GPCC_STEP_PROF   // scripts/microbench/step_prof.cu: per-warp clock() stamps of every sweep step, kept in shared memory
#define GPCC_PROF_MAXSTEPS 200
#define GPCC_STAMP(slot) do { if ((threadIdx.x & 31) == 0) prof[((slot) * 8 + (threadIdx.x >> 5)) * GPCC_PROF_MAXSTEPS + k] = (unsigned)clock(); } while (0)
#define GPCC_PROF_PARAM , unsigned* prof
#define GPCC_PROF_ARG , prof
#else
#define GPCC_STAMP(slot) do { } while (0)
#define GPCC_PROF_PARAM
#define GPCC_PROF_ARG
#endif

// ---- one sweep step -------------------------------------------------------------------------------------------------------
// A step is bound by the chain through the warp that owns the next pivot: its tile update, the reciprocal of the next pivot,
// its stores of the next column, then the barrier at which every other warp waits for it (of the ~970 cycles of a step for a
// CTA alone on its SM, the 64 DFMAs of a warp are 144 issue cycles: per-warp timelines of scripts/microbench/step_prof.cu in
// profiles/README.md).  So the step keeps that chain short:
//   * the row pair that holds the next pivot row is updated first and the reciprocal of the next pivot is formed right
//     behind it by EVERY thread, branch free (approximate reciprocal + three Newton steps, no IEEE special-case branch), so
//     that its latency hides under the remaining 48 DFMAs instead of sitting between the update and the barrier;
//   * `publish` is one branch per owner role with no warp vote and no activity flag: threads beyond the last tile have
//     out-of-range tile coordinates and own nothing;
//   * buffer parities are compile-time, and full tiles run eight steps without loop-exit tests.
__device__ __forceinline__ double fast_rcp(double d) {
    double x;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(x) : "d"(d));
    double e = fma(-d, x, 1.0);
    x = fma(x, e, x);
    e = fma(-d, x, 1.0);
    x = fma(x, e, x);
    e = fma(-d, x, 1.0);
    x = fma(x, e, x);
    return x;
}

// Publish column k+1 (tile tkn, in-tile index KKN) of the symmetric matrix, its pivot and the pivot's reciprocal prn for the
// next sweep step.  Scalar STS.64 straight from the tile registers (no staging moves).
template <int KKN>
__device__ __forceinline__ void publish(const double (&A)[8][8], int ti, int tj, int tkn, double* nb, double* pslot, double* pivslot,
                                        double prn, bool fwd) {
    const bool pc = (tj == tkn), prw = (ti == tkn) && (!fwd || pc);   // forward-only mode: the row part is never read again
    if (pc) {
        double* dst = nb + ti;
        if (prw) {  // diagonal tile: below the diagonal from the column, above it from the row
#pragma unroll
            for (int r = 0; r < 8; ++r) dst[r * CS] = (r >= KKN) ? A[r][KKN] : A[KKN][r];
            *pivslot = A[KKN][KKN];
            *pslot = prn;
        } else {
#pragma unroll
            for (int r = 0; r < 8; ++r) dst[r * CS] = A[r][KKN];
        }
    } else if (prw) {
        double* dst = nb + tj;
#pragma unroll
        for (int c = 0; c < 8; ++c) dst[c * CS] = A[KKN][c];
    }
}

template <int KK>
__device__ __forceinline__ void sweep_step(double (&A)[8][8], int ti, int tj, int tk, int k, double* cbuf, double* pbuf,
                                           double* piv, bool fwd GPCC_PROF_PARAM) {
    GPCC_STAMP(0);
    constexpr int PAR = KK & 1, NPAR = PAR ^ 1;     // k = 8 tk + KK: the buffer parity is known at compile time
    constexpr int KKN = (KK + 1) & 7;
    const bool live = !fwd || tj >= tk;
    double prn = 0.0;
    if (live) {
        const double* cb = cbuf + PAR * VLEN;
        double v[8];
        load8(cb, tj, v);
        const double pr = pbuf[PAR];
#pragma unroll
        for (int c = 0; c < 8; ++c) v[c] *= pr;
        // Column k of its owner tiles must become c * (1/d).  Those registers hold exactly the broadcast values c, so
        // running the generic update with the multiplier (1 - 1/d) in that column writes c - c (1 - 1/d) = c/d without
        // any extra instruction (relative error eps*d in entries of the inverse only; pivots, log-det and the
        // quadratic form never read the swept region).
        // Row k of its owner tiles must become c * (1/d) as well: there the registers hold c and the row multiplier is the
        // pivot d itself, so using (d - 1) instead gives c - (d - 1) c/d = c/d.  Only the diagonal element needs a fix.
        const bool own_col = (tj == tk), own_row = (ti == tk);
        if (own_col) v[KK] = 1.0 - pr;
#pragma unroll
        for (int pp = 0; pp < 4; ++pp) {
            constexpr int P0 = KKN >> 1;
            const int part = (pp + P0) & 3;          // compile-time after unrolling
            double x0 = cb[2 * part * CS + ti], x1 = cb[(2 * part + 1) * CS + ti];
            if (part == (KK >> 1) && own_row) {      // row k of its owners becomes c/d
                if (KK & 1) x1 -= 1.0; else x0 -= 1.0;
            }
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                A[2 * part][c] = fma(-x0, v[c], A[2 * part][c]);
                A[2 * part + 1][c] = fma(-x1, v[c], A[2 * part + 1][c]);
            }
            if (pp == 0) prn = fast_rcp(A[KKN][KKN]);   // final for this step; only the owner of the next pivot publishes it
        }
        if (own_col && own_row) A[KK][KK] = -pr;
    }
    GPCC_STAMP(1);
    publish<KKN>(A, ti, tj, KK < 7 ? tk : tk + 1, cbuf + NPAR * VLEN, pbuf + NPAR, piv + k + 1, prn, fwd);
    GPCC_STAMP(2);
    __syncthreads();
    GPCC_STAMP(3);
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Deterministic block sum: xor-tree inside each warp, then every thread adds the warp totals in order.
__device__ __forceinline__ double block_sum(double v, double* red, int tid, int nthreads) {
    v = warp_sum(v);
    __syncthreads();
    if ((tid & 31) == 0) red[tid >> 5] = v;
    __syncthreads();
    double s = 0.0;
    const int nw = (nthreads + 31) >> 5;
    for (int w = 0; w < nw; ++w) s += red[w];
    return s;
}

// One evaluation by the whole CTA.  `smem` is eval_smem_bytes(T, want_grad) bytes of shared memory, 16-byte aligned.
// Inputs: delays_e[L], alpha_e[L] (any address space), rho.  Outputs (written by a few threads; the caller synchronises before
// reading them): *out_ll, out_grad[L+1] (want_grad), *out_info.  Must be called by all threads of the CTA.
template <int KID>
__device__ __forceinline__ void eval_one(const DevProblem& p, int T, double* smem, const double* delays_e, const double* alpha_e,
                                         double rho, bool want_grad, bool fwd, double* out_ll, double* out_grad, int* out_info) {
    const int N = p.N, L = p.L;
    const int Np = T * TS;
    const int nthreads = blockDim.x;
    const int tid = threadIdx.x;
    const int ntiles = T * (T + 1) / 2;
    const bool active = tid < ntiles;
    // Only active threads read q.  The fallback for the others is dead code, but without it ptxas allocates the registers of
    // the 255-register fit kernels differently (spills up in four instantiations, down in four), so it stays.
    const int q = active ? tid : ntiles - 1;
    int ti, tj;
    if (!active) { ti = T; tj = T; }   // threads beyond the last tile: out-of-range coordinates, never owners of anything
    else if (fwd) {   // column-major tile order (see the header comment)
        int c = 0, rem = q;
        while (rem >= T - c) { rem -= T - c; ++c; }
        tj = c;
        ti = c + rem;
    } else {
        ti = (int)((sqrtf(8.0f * (float)q + 1.0f) - 1.0f) * 0.5f);
        while (ti * (ti + 1) / 2 > q) --ti;
        while ((ti + 1) * (ti + 2) / 2 <= q) ++ti;
        tj = q - ti * (ti + 1) / 2;
    }

    double* tsh = smem;             // shifted times t_i - tau_band(i)         (chunk layout)
    double* av = tsh + VLEN;        // alpha_band(i), 0 for padding            (chunk layout)
    double* sbv = av + VLEN;        // Sigma_b[band(i)]                         (chunk layout)
    double* dadd = sbv + VLEN;      // sigma_i^2                                (chunk layout)
    double* cbuf = dadd + VLEN;     // 2 x broadcast column                     (chunk layout; 4 VLEN reserved)
    double* piv = cbuf + 4 * VLEN;  // pivots                                   (natural)
    double* abuf = piv + VLEN;      // residual r, later a = K~^-1 r            (chunk layout)
    double* pbuf = abuf + VLEN;     // 2 pivot reciprocals (+2 pad)
    double* red = pbuf + 4;         // 64 reduction slots
    int* s_bad_p = reinterpret_cast<int*>(red + 48);
    double* part = red + 64;        // [T][T][8] gradient row-sum partials (gradient only)
    int* bandv = reinterpret_cast<int*>(part + (want_grad ? T * T * 8 : 0));  // [Np] natural

    const KernParams kp = make_kern_params(KID, rho);

    for (int i = tid; i < Np; i += nthreads) {
        const int ci = cidx(i);
        if (i < N) {
            const int bi = p.band[i];
            tsh[ci] = p.t[i] - delays_e[bi];   // delayedCovariance.jl:27 (x - delays[l])
            av[ci] = alpha_e[bi];
            sbv[ci] = p.sigb[i];
            dadd[ci] = p.s2[i];
            abuf[ci] = p.resid[i];
            bandv[i] = bi;
        } else {
            tsh[ci] = 0.0; av[ci] = 0.0; sbv[ci] = 0.0; dadd[ci] = 0.0; abuf[ci] = 0.0;
            bandv[i] = -1 - i;
        }
    }
    __syncthreads();

    // ---- assembly of the bordered matrix tile in registers --------------------------------------
    // Fully unrolled, unlike the gradient below: a rolled row loop keeps all 64 accumulators live from the first row on and
    // spills (81 against 61 us per evaluation and SM, profiles/README.md).
    double A[8][8];
    if (!active) {
#pragma unroll
        for (int r = 0; r < 8; ++r)
#pragma unroll
            for (int c = 0; c < 8; ++c) A[r][c] = 0.0;
    } else {
        double tc[8], ac[8], rc[8];
        int bc[8];
        load8(tsh, tj, tc);
        load8(av, tj, ac);
        load8(abuf, tj, rc);
#pragma unroll
        for (int c = 0; c < 8; ++c) bc[c] = bandv[tj * 8 + c];
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            const int i = ti * 8 + r;
            const int ci = cidx(i);
            const double tr = tsh[ci], ar = av[ci], sbr = sbv[ci], dr = dadd[ci];
            const int br = bandv[i];
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const int j = tj * 8 + c;
                const double kv = kern_value<KID>(tr - tc[c], kp);
                double val = (ar * ac[c]) * kv;          // scale[l]*scale[m]*kernel  (delayedCovariance.jl:27)
                if (i == j) val += dr;                   // + Sobs                   (gpccfixdelay_marginaliseb.jl:135)
                if (br == bc[c]) val += sbr;             // + B = Q Sigma_b Q'
                if (i == N) val = rc[c];                 // border row: r = Y - bbar (corner = 0)
                if (i > N && i == j) val = 1.0;          // padding
                A[r][c] = val;
            }
        }
    }
    __syncthreads();   // everyone has read abuf/tsh before cbuf traffic starts (abuf is reused later)

    // ---- publish column 0, then N sweep steps ----------------------------------------------------
#ifdef GPCC_STEP_PROF
    __shared__ unsigned prof[4 * 8 * GPCC_PROF_MAXSTEPS];
#endif
    publish<0>(A, ti, tj, 0, cbuf, pbuf, piv, fast_rcp(A[0][0]), fwd);
    __syncthreads();
    for (int tk = 0; 8 * tk < N; ++tk) {   // one copy of the eight specialised steps; the guards only matter in the last tile
        const int k0 = tk * 8;               // (the last step also publishes "column N", the border row: never read, harmless)
        sweep_step<0>(A, ti, tj, tk, k0 + 0, cbuf, pbuf, piv, fwd GPCC_PROF_ARG);
        if (k0 + 1 < N) sweep_step<1>(A, ti, tj, tk, k0 + 1, cbuf, pbuf, piv, fwd GPCC_PROF_ARG);
        if (k0 + 2 < N) sweep_step<2>(A, ti, tj, tk, k0 + 2, cbuf, pbuf, piv, fwd GPCC_PROF_ARG);
        if (k0 + 3 < N) sweep_step<3>(A, ti, tj, tk, k0 + 3, cbuf, pbuf, piv, fwd GPCC_PROF_ARG);
        if (k0 + 4 < N) sweep_step<4>(A, ti, tj, tk, k0 + 4, cbuf, pbuf, piv, fwd GPCC_PROF_ARG);
        if (k0 + 5 < N) sweep_step<5>(A, ti, tj, tk, k0 + 5, cbuf, pbuf, piv, fwd GPCC_PROF_ARG);
        if (k0 + 6 < N) sweep_step<6>(A, ti, tj, tk, k0 + 6, cbuf, pbuf, piv, fwd GPCC_PROF_ARG);
        if (k0 + 7 < N) sweep_step<7>(A, ti, tj, tk, k0 + 7, cbuf, pbuf, piv, fwd GPCC_PROF_ARG);
    }

#ifdef GPCC_STEP_PROF
    if (blockIdx.x == gpcc_prof_block)
        for (int i = tid; i < 4 * 8 * GPCC_PROF_MAXSTEPS; i += nthreads) gpcc_prof_out[i] = prof[i];
#endif
    // ---- log-determinant, info, quadratic form ---------------------------------------------------
    const int tN = N >> 3, rN = N & 7;
    double ld = 0.0;
    int bad = INT_MAX;
    for (int k = tid; k < N; k += nthreads) {
        const double d = piv[k];
        if (!(d > 0.0)) bad = min(bad, k + 1); else ld += log(d);
    }
    ld = block_sum(ld, red, tid, nthreads);
    if (tid == 0) *s_bad_p = INT_MAX;
    __syncthreads();
    if (bad != INT_MAX) atomicMin(s_bad_p, bad);   // min is order independent: deterministic
    __syncthreads();
    const int info = (*s_bad_p == INT_MAX) ? 0 : *s_bad_p;

    if (active && ti == tN && tj == tN) {
        double qv = 0.0;
#pragma unroll
        for (int r = 0; r < 8; ++r) if (r == rN) qv = -A[r][r];
        red[32] = qv;
    }
    __syncthreads();
    const double quad = red[32];
    const double ll = -0.5 * ((double)N * LOG2PI + ld + quad);   // logpdf(MvNormal(bbar,K), Y)  (:139)
    if (tid == 0) {
        *out_ll = info ? -INFINITY : ll;
        *out_info = info;
    }
    if (!want_grad) return;
    if (info) {
        if (tid <= L) out_grad[tid] = 0.0;
        return;
    }

    // ---- gradient: W = a a' - K~^-1 contracted with K and dK/drho (full sweep only: fwd is false here) -----------
    if (active && ti == tN) {   // border row holds a = K~^-1 r
        double vals[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            double x = 0.0;
#pragma unroll
            for (int r = 0; r < 8; ++r) if (r == rN) x = A[r][c];
            vals[c] = (tj * 8 + c < N) ? x : 0.0;
        }
        store8(abuf, tj, vals);
    }
    __syncthreads();

    // Two forms of the same sums, selected per translation unit.  The rolled one (GPCC_ROLL_GRADIENT, defined by small_fit.cu)
    // takes the row of the tile out of its registers through a switch with static indices: one copy of the four kernel
    // evaluations instead of 32.  The persistent fit kernel's CTAs drift apart, two co-resident CTAs are in different phases,
    // and the smaller instruction footprint measured 2 % faster there (profiles/README.md).  In the batch kernel the rolled
    // form changes the register allocation of the whole kernel, and forward-only evaluations, which never reach this code,
    // measured 0.7 % slower at N = 150; so small_sweep.cu keeps the unrolled form.
#ifdef GPCC_ROLL_GRADIENT
    double es = 0.0;
    const bool diag_tile = (ti == tj);
    double* myrow = part + (ti * T + tj) * 8;       // row sums of this tile, [8]
#pragma unroll
    for (int half = 0; half < 2; ++half) {           // four columns at a time: limits the live column data
        double tc[4], ac[4], wc[4], cols[4];
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) {
            const int cj = cidx(tj * 8 + half * 4 + cc);
            tc[cc] = tsh[cj]; ac[cc] = av[cj]; wc[cc] = abuf[cj]; cols[cc] = 0.0;
        }
#pragma unroll 1
        for (int r = 0; r < 8; ++r) {
            const int ci = cidx(ti * 8 + r);
            const double tr = tsh[ci], ar = av[ci], wr = abuf[ci];
            double ain[4];
#define GPCC_ROW_OUT(R) case R: _Pragma("unroll") for (int cc = 0; cc < 4; ++cc) ain[cc] = A[R][half * 4 + cc]; break;
            switch (r) { GPCC_ROW_OUT(0) GPCC_ROW_OUT(1) GPCC_ROW_OUT(2) GPCC_ROW_OUT(3) GPCC_ROW_OUT(4) GPCC_ROW_OUT(5) GPCC_ROW_OUT(6) default: _Pragma("unroll") for (int cc = 0; cc < 4; ++cc) ain[cc] = A[7][half * 4 + cc]; break; }
#undef GPCC_ROW_OUT
            double rsum = 0.0;
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) {
                const int c = half * 4 + cc;
                const double W = fma(wr, wc[cc], ain[cc]);        // a_i a_j - (K~^-1)_ij
                double kv, dkv;
                kern_value_drho<KID>(tr - tc[cc], kp, kv, dkv);
                const double aa = ar * ac[cc];                   // 0 on padding / border rows
                double ct = W * (aa * kv);
                double et = W * (aa * dkv);
                if (diag_tile) {
                    if (r == c) { rsum += ct; ct = 0.0; et = 0.0; }      // diagonal counted once, dk(0)=0
                    else if (r < c) { ct = 0.0; et = 0.0; }              // upper part of the tile is unused
                }
                rsum += ct;
                cols[cc] += ct;
                es += et;
            }
            if (active) { if (half == 0) myrow[r] = rsum; else myrow[r] += rsum; }
        }
        if (active && !diag_tile) {
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) part[(tj * T + ti) * 8 + half * 4 + cc] = cols[cc];
        }
        if (active && diag_tile) {
            // fold the column sums of the strictly-lower part into the same slots as the row sums (the slots belong to this
            // thread alone, so the later "+=" of the second half simply adds on top)
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) myrow[half * 4 + cc] += cols[cc];
        }
    }
#else
    double rows[8];
#pragma unroll
    for (int r = 0; r < 8; ++r) rows[r] = 0.0;
    double es = 0.0;
    const bool diag_tile = (ti == tj);
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        double tc[4], ac[4], wc[4], cols[4];
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) {
            const int cj = cidx(tj * 8 + half * 4 + cc);
            tc[cc] = tsh[cj]; ac[cc] = av[cj]; wc[cc] = abuf[cj]; cols[cc] = 0.0;
        }
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            const int ci = cidx(ti * 8 + r);
            const double tr = tsh[ci], ar = av[ci], wr = abuf[ci];
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) {
                const int c = half * 4 + cc;
                const double W = fma(wr, wc[cc], A[r][c]);       // a_i a_j - (K~^-1)_ij
                double kv, dkv;
                kern_value_drho<KID>(tr - tc[cc], kp, kv, dkv);
                const double aa = ar * ac[cc];                   // 0 on padding / border rows
                double ct = W * (aa * kv);
                double et = W * (aa * dkv);
                if (diag_tile) {
                    if (r == c) { rows[r] += ct; ct = 0.0; et = 0.0; }   // diagonal counted once, dk(0)=0
                    else if (r < c) { ct = 0.0; et = 0.0; }              // upper part of the tile is unused
                }
                rows[r] += ct;
                cols[cc] += ct;
                es += et;
            }
        }
        if (active) {
            if (!diag_tile) {
#pragma unroll
                for (int cc = 0; cc < 4; ++cc) part[(tj * T + ti) * 8 + half * 4 + cc] = cols[cc];
            } else {
                // fold the column sums of the strictly-lower part into the same slot as the row sums
#pragma unroll
                for (int cc = 0; cc < 4; ++cc) {
#pragma unroll
                    for (int r = 0; r < 8; ++r) if (r == half * 4 + cc) rows[r] += cols[cc];
                }
            }
        }
    }
    if (active) {
#pragma unroll
        for (int r = 0; r < 8; ++r) part[(ti * T + tj) * 8 + r] = rows[r];
    }
#endif
    es = block_sum(active ? es : 0.0, red, tid, nthreads);   // (contains the __syncthreads that orders `part`)

    // s_i = sum_j W_ij K_ij (full row);  dlogL/dalpha_p = (1/alpha_p) sum_{i in band p} s_i
    double* srow = cbuf;   // natural layout, reuse
    for (int i = tid; i < N; i += nthreads) {
        const double* pp = part + (size_t)(i >> 3) * T * 8 + (i & 7);
        double s = 0.0;
        for (int src = 0; src < T; ++src) s += pp[src * 8];
        srow[i] = s;
    }
    __syncthreads();
    const int warp = tid >> 5, lane = tid & 31, nwarps = (nthreads + 31) >> 5;
    for (int pb = warp; pb < L; pb += nwarps) {
        double s = 0.0;
        for (int i = p.band_start[pb] + lane; i < p.band_start[pb + 1]; i += 32) s += srow[i];
        s = warp_sum(s);
        if (lane == 0) out_grad[pb] = s / alpha_e[pb];
    }
    if (tid == 0) out_grad[L] = es;   // 0.5 * sum_full = sum over the strict lower triangle
}

}  // namespace small
}  // namespace gpcc
