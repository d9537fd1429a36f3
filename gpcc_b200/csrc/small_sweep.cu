// Batch form of the fused small-N evaluator: one CTA per (delay candidate, hyper-parameter) pair (small_eval.cuh has the
// design).  Serves gpcc_loglik_batch / gpcc_loglik_theta_batch and the host-driven L-BFGS; the fitted grid itself runs in
// the persistent kernel of small_fit.cu.
#include "small_eval.cuh"
#include <cstdlib>

namespace gpcc {
namespace {

using namespace small;

template <int KID, int MAXTHREADS, int MINBLOCKS>
__global__ void __launch_bounds__(MAXTHREADS, MINBLOCKS)
small_sweep_kernel(DevProblem p, EvalBatch b, int T, int fwd) {
    extern __shared__ __align__(16) double smem[];
    const int e = blockIdx.x;
    eval_one<KID>(p, T, smem, b.delays + (size_t)e * p.L, b.alpha + (size_t)e * p.L, b.rho[e], b.want_grad != 0, fwd != 0,
                  b.ll + e, b.grad + (size_t)e * (p.L + 1), b.info + e);
}

template <int KID, int MT, int MB>
void go(const DevProblem& p, const EvalBatch& b, int T, int threads, int maxT, int fwd, cudaStream_t s) {
    auto kfn = small_sweep_kernel<KID, MT, MB>;
    cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)eval_smem_bytes(maxT, 1));
    kfn<<<b.M, threads, eval_smem_bytes(T, b.want_grad), s>>>(p, b, T, fwd);
}

template <int KID>
cudaError_t launch_kid(const DevProblem& p, const EvalBatch& b, int T, cudaStream_t s) {
    const int ntiles = T * (T + 1) / 2;
    const int threads = (ntiles + 31) / 32 * 32;
    static const int variant_env = getenv("GPCC_SMALL_VARIANT") ? atoi(getenv("GPCC_SMALL_VARIANT")) : -1;
    static int nsm = 0;
    if (nsm == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
    }
    // Occupancy variant by batch size (measured on B200, profiles/small_sweep_variants_r1.log).
    //   N <= 119 (T <= 15: 120 tiles, 128 threads): three CTAs per SM are 8 % faster once every SM has three (32.7 vs
    //   35.6 us per evaluation and SM), but slower when the batch leaves SMs with one or two (82 vs 65 us at one CTA per SM);
    //   N <= 151 (192 threads): a CTA that is alone on its SM runs faster with 255 registers and no spills (101 vs 122 us),
    //   two co-resident CTAs at 168 registers win as soon as there is more than one evaluation per SM (134 vs 188 us for two).
    int variant = variant_env;
    if (variant < 0) variant = (threads <= 128) ? (b.M >= 3 * nsm ? 2 : 1) : (b.M <= nsm ? 0 : 1);
    // forward-only mode (N^3/3 flop) when no gradient is wanted
    const int fwd = b.want_grad ? 0 : 1;
    if (threads <= 128) {
        if (variant == 2) go<KID, 128, 3>(p, b, T, threads, 15, fwd, s);
        else              go<KID, 128, 2>(p, b, T, threads, 15, fwd, s);
    } else if (threads <= 192 && variant == 1) go<KID, 192, 2>(p, b, T, threads, 19, fwd, s);
    else if (threads <= 224)                   go<KID, 224, 1>(p, b, T, threads, 20, fwd, s);
    else                                       go<KID, 352, 1>(p, b, T, threads, SMALL_MAX_T, fwd, s);
    return cudaGetLastError();
}

}  // namespace

// One kernel family per object file (compiled four times with -DGPCC_KID=0..3); small_dispatch.cu selects by kernel id.
#define GPCC_CAT2(a, b) a##b
#define GPCC_CAT(a, b) GPCC_CAT2(a, b)
cudaError_t GPCC_CAT(small_sweep_launch_k, GPCC_KID)(const DevProblem& p, const EvalBatch& b, cudaStream_t s) {
    const int T = (p.N + 1 + SMALL_TILE - 1) / SMALL_TILE;
    return launch_kid<GPCC_KID>(p, b, T, s);
}

}  // namespace gpcc
