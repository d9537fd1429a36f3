// Device-resident fit of the fused small-N path: getsolution (src/gpccfixdelay_marginaliseb.jl:203-215) for a whole grid of
// delay candidates in ONE kernel launch.
//
// A persistent CTA takes the next candidate from an atomic work queue and runs, without leaving the kernel,
//   screening   the P (`initialrandom`) start points theta0 (:207-209), forward-only evaluations (N^3/3 flop each),
//               first minimum wins (Julia `argmin`),
//   start       logL + analytic gradient at the winner,
//   L-BFGS      the state machine of lbfgs.h (the one the host-driven driver uses), state in shared memory, thread 0
//               does the O(history * L) update between two evaluations while the second resident CTA keeps the SM busy,
// with the (N+1) x (N+1) bordered matrix of every evaluation in the registers of the CTA (small_eval.cuh).
// Compared with the host-driven batched loop (api.cu, fit_shard) this removes ~220 kernel launches, H2D/D2H copies and
// host synchronisations per fitted grid, the straggler tail of the batched rounds (a round ends when its slowest
// candidate ends; here a slow candidate only occupies its own CTA) and the host threads that contend when 8 ranks share
// one box.  Results do not depend on the schedule: candidates never interact.
// The gradient phase is compiled in its rolled form here (one copy of the kernel evaluations instead of 32): the CTAs of the
// persistent kernel drift apart, two co-resident CTAs are usually in different phases, and the smaller instruction footprint
// measured 2 % faster (profiles/README.md); in the batch kernel, whose CTAs run in step, it is neutral.
#define GPCC_ROLL_GRADIENT
#include "small_eval.cuh"
#include "lbfgs.h"
#include "nm.h"
#include <cstdlib>

namespace gpcc {
namespace {

using namespace small;

struct FitCtl {                 // per-CTA control block in shared memory
    LbfgsState S;
    NmState NM;                 // optimizer = 1 only
    double delays[MAX_BANDS];
    double alpha[MAX_BANDS];    // constrained parameters of the evaluation in flight
    double rho;
    double jac[LBFGS_MAXN];     // d(alpha, rho)/d theta at the evaluation in flight
    double theta_next[LBFGS_MAXN];   // unconstrained parameters of the next evaluation (unpacked by L+1 threads)
    double theta_best[LBFGS_MAXN];
    double res_ll;
    double res_grad[LBFGS_MAXN];
    double bestf;
    int res_info;
    int cand, phase, j, best, want_grad, fwd;
    unsigned n_grad, n_fwd;
};
enum { PH_SCREEN = 0, PH_START = 1, PH_LBFGS = 2, PH_DONE = 3, PH_NM = 4 };

__device__ __forceinline__ double softplus(double x) { return x > 0 ? x + log1p(exp(-x)) : log1p(exp(x)); }
__device__ __forceinline__ double logistic(double x) { return 0.5 * (1.0 + tanh(0.5 * x)); }

// unpack (gpccfixdelay_marginaliseb.jl:112-126): alpha = makepositive(theta_l) + floor, rho = transformbetween(theta_L+1).
// One thread per parameter: the FP64 exp / log1p / tanh chains of the L+1 transforms run side by side instead of one after
// the other on thread 0 (the profile showed the other five warps waiting ~9 % of the kernel time for that thread).
__device__ __forceinline__ void unpack_to_ctl(FitCtl& c, const double* theta, int, const FitParams&) {
    for (int k = 0; k < c.S.n; ++k) c.theta_next[k] = theta[k];
}
__device__ __forceinline__ void unpack_parallel(FitCtl& c, int tid, int L, const FitParams& fp) {
    if (tid < L) {
        c.alpha[tid] = softplus(c.theta_next[tid]) + fp.alpha_floor;
        c.jac[tid] = logistic(c.theta_next[tid]);
    } else if (tid == L) {
        const double s = logistic(c.theta_next[L]);
        c.rho = fp.rhomin + (fp.rhomax - fp.rhomin) * s;
        c.jac[L] = (fp.rhomax - fp.rhomin) * s * (1.0 - s);
    }
}

// Thread 0: consume the result of the evaluation that just finished (if any) and set up the next one, or finish.
// OPT is a template parameter so that the Nelder-Mead code does not weigh on the registers of the default (L-BFGS) kernel.
template <int OPT>
__device__ void advance(FitCtl& c, int L, const FitParams& fp, const FitBuffers& fb, const LbfgsOptions& lo) {
    const int n = L + 1;
    const double* th0 = fb.theta0 + (fp.theta0_per_candidate ? (size_t)c.cand * fp.P * n : 0);
    if (c.phase == PH_SCREEN) {
        if (c.j > 0) {                                    // result of start point j-1
            const double f = -c.res_ll;
            if (c.res_info == 0 && lb_finite(f) && f < c.bestf) {   // first minimum wins (Julia argmin, :209)
                c.bestf = f;
                c.best = c.j - 1;
            }
        }
        if (c.j < fp.P) {
            unpack_to_ctl(c, th0 + (size_t)c.j * n, L, fp);
            c.want_grad = 0; c.fwd = 1; ++c.n_fwd;
            ++c.j;
            return;
        }
        c.S.n = n;
        c.S.nfev = fp.P;
        c.S.iters = 0;
        if (c.best < 0) { c.S.status = LbfgsState::NO_START; c.S.f = lb_inf(); c.phase = PH_DONE; return; }
        lb_copy(c.theta_best, th0 + (size_t)c.best * n, n);
        if (fp.max_iter <= 0) {                           // screening only (:207-209): no gradient is needed
            lb_copy(c.S.x, c.theta_best, n);
            c.S.f = c.bestf; c.S.status = LbfgsState::ITER_CAP; c.phase = PH_DONE;
            return;
        }
        if (OPT == 1) {                                   // the reference's Nelder-Mead (:205-211): forward-only evaluations
            c.NM.start(n, c.theta_best, c.bestf, fp.max_iter, fp.nm_gtol);
            c.phase = PH_NM;
            if (c.NM.phase != NmState::DONE) {
                unpack_to_ctl(c, c.NM.xt, L, fp);
                c.want_grad = 0; c.fwd = 1; ++c.n_fwd;
                return;
            }
        } else {                                          // gradient at the winner only
            unpack_to_ctl(c, c.theta_best, L, fp);
            c.want_grad = 1; c.fwd = 0; ++c.n_grad;
            c.phase = PH_START;
            return;
        }
    } else if (OPT == 1 && c.phase == PH_NM) {                        // result at NM.xt
        c.NM.feed(c.res_info == 0 && lb_finite(c.res_ll), -c.res_ll, fp.max_iter, fp.nm_gtol);
        if (c.NM.phase != NmState::DONE) {
            unpack_to_ctl(c, c.NM.xt, L, fp);
            c.want_grad = 0; c.fwd = 1; ++c.n_fwd;
            return;
        }
    } else if (c.phase == PH_START) {
        double g[LBFGS_MAXN];
        for (int k = 0; k < n; ++k) g[k] = -c.res_grad[k] * c.jac[k];
        c.S.start(n, c.theta_best, c.bestf, g, lo);       // the forward-only value and the sweep's value are the same bits
    } else {                                              // PH_LBFGS: result at S.xt
        const bool ok = c.res_info == 0 && lb_finite(c.res_ll);
        double g[LBFGS_MAXN];
        for (int k = 0; k < n; ++k) g[k] = ok ? -c.res_grad[k] * c.jac[k] : 0.0;
        c.S.feed(ok, -c.res_ll, g, lo);
    }
    if (OPT == 1 && c.phase == PH_NM) {                   // Nelder-Mead finished: report through the common fields
        c.S.f = c.NM.fbest;
        lb_copy(c.S.x, c.NM.xbest, n);
        c.S.iters = c.NM.iters;
        c.S.nfev = fp.P + c.NM.nfev;
        c.S.status = c.NM.status;
        c.phase = PH_DONE;
        return;
    }
    if (c.S.status != LbfgsState::RUNNING) { c.phase = PH_DONE; return; }
    c.phase = PH_LBFGS;
    unpack_to_ctl(c, c.S.xt, L, fp);
    c.want_grad = 1; c.fwd = 0; ++c.n_grad;
}

template <int KID, int MAXTHREADS, int MINBLOCKS, int OPT>
__global__ void __launch_bounds__(MAXTHREADS, MINBLOCKS)
small_fit_kernel(DevProblem p, FitParams fp, FitBuffers fb, int T, int ctl_offset_doubles) {
    extern __shared__ __align__(16) double smem[];
    FitCtl& c = *reinterpret_cast<FitCtl*>(smem + ctl_offset_doubles);
    const int tid = threadIdx.x, L = p.L, n = L + 1;
    LbfgsOptions lo;
    lo.max_iter = fp.max_iter; lo.gtol = fp.gtol; lo.ftol = fp.ftol; lo.history = fp.history; lo.n_scale = L;
    if (tid == 0) {                                        // schedule diagnostics: when did the first CTA start
        unsigned long long t0;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
        atomicMin(fb.counters + 5, t0);
    }
    for (;;) {
        __syncthreads();                                   // the previous candidate's control block is no longer read
        if (tid == 0) {
            const unsigned long long qpos = atomicAdd(fb.counters, 1ULL);
            c.cand = qpos < (unsigned long long)fp.M ? fb.order[qpos] : fp.M;
            c.phase = PH_SCREEN; c.j = 0; c.best = -1; c.bestf = lb_inf(); c.S.n = n;
            c.n_grad = 0; c.n_fwd = 0;
        }
        __syncthreads();
        const int cand = c.cand;
        if (cand >= fp.M) break;
        if (tid < L) c.delays[tid] = fb.delays[(size_t)cand * L + tid];
        for (;;) {
            if (tid == 0) {
#ifdef GPCC_FIT_PROF
                const long long ta = clock64();
#endif
                advance<OPT>(c, L, fp, fb, lo);
#ifdef GPCC_FIT_PROF
                atomicAdd(fb.counters + 7, (unsigned long long)(clock64() - ta));
#endif
            }
            __syncthreads();
            if (c.phase == PH_DONE) break;
            if (tid <= L) unpack_parallel(c, tid, L, fp);
            __syncthreads();
            eval_one<KID>(p, T, smem, c.delays, c.alpha, c.rho, c.want_grad != 0, c.fwd != 0, &c.res_ll, c.res_grad, &c.res_info);
            __syncthreads();
        }
        if (tid == 0) {
            fb.ll[cand] = -c.S.f;                          // -result.minimum (:351)
            fb.iters[cand] = c.S.iters;
            fb.nfev[cand] = c.S.nfev;
            fb.status[cand] = c.S.status;
            atomicAdd(fb.counters + 1, (unsigned long long)c.n_grad);
            atomicAdd(fb.counters + 2, (unsigned long long)c.n_fwd);
        }
        if (tid < n) fb.theta[(size_t)cand * n + tid] = (c.S.status == LbfgsState::NO_START) ? nan("") : c.S.x[tid];
    }
    if (tid == 0) {                                        // ... and when did this CTA run out of work (sum and max over CTAs)
        unsigned long long t1;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
        atomicAdd(fb.counters + 3, t1 - fb.counters[5]);
        atomicMax(fb.counters + 4, t1);
        atomicAdd(fb.counters + 6, 1ULL);
    }
}

template <int KID, int MT, int MB, int OPT>
cudaError_t go2(const DevProblem& p, const FitParams& fp, const FitBuffers& fb, int T, int threads, int maxT, int nsm, cudaStream_t s) {
    auto kfn = small_fit_kernel<KID, MT, MB, OPT>;
    const size_t ev = (eval_smem_bytes(T, 1) + 15) / 16 * 16;
    const size_t ev_max = (eval_smem_bytes(maxT, 1) + 15) / 16 * 16;
    cudaError_t e = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(ev_max + sizeof(FitCtl)));
    if (e != cudaSuccess) return e;
    int per_sm = MB;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kfn, threads, ev + sizeof(FitCtl));
    if (e != cudaSuccess) return e;
    if (per_sm < 1) per_sm = 1;
    const int grid = (int)std::min<long long>(fp.M, (long long)nsm * per_sm);
    kfn<<<grid, threads, ev + sizeof(FitCtl), s>>>(p, fp, fb, T, (int)(ev / 8));
    return cudaGetLastError();
}

template <int KID, int MT, int MB>
cudaError_t go(const DevProblem& p, const FitParams& fp, const FitBuffers& fb, int T, int threads, int maxT, int nsm, cudaStream_t s) {
    if (fp.optimizer == 1) return go2<KID, MT, MB, 1>(p, fp, fb, T, threads, maxT, nsm, s);
    return go2<KID, MT, MB, 0>(p, fp, fb, T, threads, maxT, nsm, s);
}

template <int KID>
cudaError_t launch_kid(const DevProblem& p, const FitParams& fp, const FitBuffers& fb, int T, cudaStream_t s) {
    const int ntiles = T * (T + 1) / 2;
    const int threads = (ntiles + 31) / 32 * 32;
    int dev = 0, nsm = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
    // occupancy variants as in small_sweep.cu: more co-resident CTAs at 168 registers once every SM gets that many
    if (threads <= 128) {
        if (fp.M >= 3 * nsm) return go<KID, 128, 3>(p, fp, fb, T, threads, 15, nsm, s);
        return go<KID, 128, 2>(p, fp, fb, T, threads, 15, nsm, s);
    }
    if (threads <= 192 && fp.M > nsm) return go<KID, 192, 2>(p, fp, fb, T, threads, 19, nsm, s);
    if (threads <= 224) return go<KID, 224, 1>(p, fp, fb, T, threads, 20, nsm, s);
    return go<KID, 352, 1>(p, fp, fb, T, threads, SMALL_MAX_T, nsm, s);
}

}  // namespace

// One kernel family per object file (the Makefile compiles this source four times with -DGPCC_KID=0..3 so that the
// instantiations build in parallel); small_dispatch.cu selects by kernel id.
#define GPCC_CAT2(a, b) a##b
#define GPCC_CAT(a, b) GPCC_CAT2(a, b)
cudaError_t GPCC_CAT(small_fit_launch_k, GPCC_KID)(const DevProblem& p, const FitParams& fp, const FitBuffers& fb, cudaStream_t s) {
    const int T = (p.N + 1 + SMALL_TILE - 1) / SMALL_TILE;
    return launch_kid<GPCC_KID>(p, fp, fb, T, s);
}

}  // namespace gpcc
