// Internal declarations shared by the CUDA translation units of libgpcc_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <string>
#include <vector>

namespace gpcc {

constexpr int MAX_BANDS = 8;   // == GPCC_MAX_BANDS

// Problem data resident on one device (uploaded once by gpcc_problem_create).
struct DevProblem {
    int N = 0;            // total points
    int L = 0;            // bands
    int kernel_id = 0;
    const double* t = nullptr;      // [N] observation times, bands concatenated
    const double* resid = nullptr;  // [N] Y - bbar            (gpccfixdelay_marginaliseb.jl:85,98)
    const double* y = nullptr;      // [N] Y                   (:85; right-hand side of the postb solve, :250)
    const double* s2 = nullptr;     // [N] sigma^2  (Sobs)     (:89)
    const double* sigb = nullptr;   // [N] Sigma_b[band(i)]    (:94-96, B = Q Sigma_b Q')
    const int* band = nullptr;      // [N] band index of point i
    int band_start[9] = {0};        // band l occupies [band_start[l], band_start[l+1])
};

// One batch of (delay, hyper-parameter) evaluations, all arrays on the device.
struct EvalBatch {
    int M = 0;
    const double* delays = nullptr;  // [M][L]
    const double* alpha = nullptr;   // [M][L]
    const double* rho = nullptr;     // [M]
    int want_grad = 0;
    double* ll = nullptr;            // [M]
    double* grad = nullptr;          // [M][L+1]
    int* info = nullptr;             // [M]
    int mode_postb = 0;              // 1 (tiled path only): factor Sobs + K WITHOUT B (the fitted state of postb / pred, :241-250)
    // host mirrors of delays / alpha / rho (optional): the tiled path compares consecutive evaluations on the host to find runs
    // that share the hyper-parameters and the delays of all bands but the last (structure reuse, large_path.cu)
    const double* h_delays = nullptr;
    const double* h_alpha = nullptr;
    const double* h_rho = nullptr;
    double* dump_chol = nullptr;     // optional [M][N*N] dense column-major Cholesky factor (lower, upper part zero); tiled path,
                                     // forward mode only (the fitted state behind postb / pred, fitstate.cu)
};

// ---- small-N path: fused register-resident symmetric sweep (small_sweep.cu) -------------------
// Largest N the fused kernel handles (N+1 padded to a multiple of 8 gives <= SMALL_MAX_T tile rows).
constexpr int SMALL_TILE = 8;
constexpr int SMALL_MAX_T = 25;
inline bool small_path_supports(int N) { return (N + 1 + SMALL_TILE - 1) / SMALL_TILE <= SMALL_MAX_T; }
cudaError_t small_sweep_launch(const DevProblem& p, const EvalBatch& b, cudaStream_t stream);

// ---- device-resident fit of the fused small-N path (small_fit.cu): screening + L-BFGS without leaving the kernel ----
struct FitParams {            // keyword arguments / constants of gpcc (gpccfixdelay_marginaliseb.jl:46, :112, :205)
    int M = 0;                // candidates of this launch
    int P = 0;                // start points per candidate (`initialrandom`)
    int theta0_per_candidate = 0;
    int max_iter = 1000;
    double rhomin = 0.1, rhomax = 20.0, alpha_floor = 1e-8, gtol = 1e-7, ftol = 1e-13;
    int history = 8;
    int optimizer = 0;        // 0: L-BFGS on the analytic gradient; 1: Nelder-Mead (nm.h), forward-only evaluations
    double nm_gtol = 1e-6;    // Optim.Options(g_tol = 1e-6) (:205)
};
struct FitBuffers {           // all on the device
    const double* delays = nullptr;   // [M][L]
    const double* theta0 = nullptr;   // [P][L+1] or [M][P][L+1]
    const int* order = nullptr;       // [M] work-queue order: position q of the queue is candidate order[q]
    double* ll = nullptr;             // [M]  -result.minimum (:351)
    double* theta = nullptr;          // [M][L+1]
    int* iters = nullptr;             // [M]
    int* nfev = nullptr;              // [M]  objective evaluations as the optimiser counts them
    int* status = nullptr;            // [M]  LbfgsState::Status
    unsigned long long* counters = nullptr;   // [8]: [0] work queue head, [1] evaluations with gradient, [2] forward-only evaluations,
                                              // [3] sum over CTAs of (exit - first start) ns, [4] last exit, [5] first start, [6] CTAs
};
cudaError_t small_fit_launch(const DevProblem& p, const FitParams& fp, const FitBuffers& fb, cudaStream_t stream);

// ---- large-N path: tiled matrix in HBM, blocked sweep with DMMA trailing updates (large_path.cu) --
struct LargeWorkspace {
    void* impl = nullptr;
};
struct LargeTimings {
    double ms_assembly = 0, ms_factor = 0, ms_gradreduce = 0;
    long long launches = 0;
    long long shared_prefix_evals = 0;   // evaluations whose leading block was factorised by another matrix of their wave
    long long assembly_bytes = 0;        // HBM bytes moved by the covariance assembly kernels (tiles written; cache imports read + written)
    long long tau_cache_evals = 0;       // evaluations that imported the band-1 steps of their last band from the last-band cache
};
cudaError_t large_eval(const DevProblem& p, const EvalBatch& b, LargeWorkspace& ws, cudaStream_t stream, bool profile,
                       LargeTimings* timings);
void large_workspace_release(LargeWorkspace& ws);

// ---- posterior over candidates (posterior.cu): src/getprobabilities.jl:10-20 --------------------
cudaError_t posterior_launch(int M, const double* d_ll, const double* d_logprior, double* d_out, cudaStream_t stream,
                             bool joint_already = false);
// sharded form: every device reduces its own slice to (max, sum exp) before the all-gather, the combine after it is G elements
//   send  [per][rec] records with the joint log-density in column `jcol`, followed by 2 doubles for the partials
cudaError_t posterior_partial_launch(int per, int rec, int jcol, double* d_send, cudaStream_t stream);
//   recv  G blocks of (per*rec + 2) doubles as gathered; out[g*per + k] = exp(joint - logsumexp)
cudaError_t posterior_combine_launch(int G, int per, int rec, int jcol, const double* d_recv, double* d_out, cudaStream_t stream);

// ---- NCCL, loaded at run time so that single-GPU use needs no NCCL at all (nccl_bridge.cpp) -------
struct NcclBridge;
NcclBridge* nccl_bridge_create(const std::vector<int>& devs, std::string& err);
int nccl_bridge_unique_id(char* out128, std::string& err);
NcclBridge* nccl_bridge_create_rank(int dev, int world, int rank, const char* id128, std::string& err);
void nccl_bridge_destroy(NcclBridge* b);
int nccl_bridge_allgather(NcclBridge* b, const std::vector<double*>& send, const std::vector<double*>& recv, int count,
                          const std::vector<cudaStream_t>& streams, std::string& err);

}  // namespace gpcc

struct gpcc_ctx;
namespace gpcc {
struct GatherIO {      // per-candidate outputs of a grid fit, host arrays of the caller (any may be NULL except ll)
    double *ll, *theta, *alpha, *rho;
    int *nfev, *info;
};
int posterior_on_devices(gpcc_ctx* ctx, int L, int M, const GatherIO& io, const double* logprior, double* out_post);
}
