// Batch form of the fused small-N evaluator: one CTA per (delay candidate, hyper-parameter) pair (small_eval.cuh has the
// design).  Serves gpcc_loglik_batch / gpcc_loglik_theta_batch and the host-driven L-BFGS; the fitted grid itself runs in
// the persistent kernel of small_fit.cu.
#include "small_eval.cuh"

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

template <int KID>
cudaError_t launch_kid(const DevProblem& p, const EvalBatch& b, int T, cudaStream_t s) {
    int dev = 0, nsm = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
    const int fwd = b.want_grad ? 0 : 1;   // forward-only mode (N^3/3 flop) when no gradient is wanted
    return with_instantiation(T, b.M, nsm, [&](auto mt, auto mb, int threads, int maxT) {
        auto kfn = small_sweep_kernel<KID, decltype(mt)::value, decltype(mb)::value>;
        const cudaError_t e = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)eval_smem_bytes(maxT, 1));
        if (e != cudaSuccess) return e;
        kfn<<<b.M, threads, eval_smem_bytes(T, b.want_grad), s>>>(p, b, T, fwd);
        return cudaGetLastError();
    });
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
