// Shared host-side state of libgpcc_b200.so (contexts, problems, per-device staging).
#pragma once
#include "../../include/gpcc_b200.h"
#include "gpcc_internal.h"
#include <algorithm>
#include <string>
#include <vector>

namespace gpcc {

int fail(int code, const std::string& msg);
const std::string& last_error();

#define CUDA_TRY(expr)                                                                            \
    do {                                                                                          \
        cudaError_t _e = (expr);                                                                  \
        if (_e != cudaSuccess) {                                                                  \
            cudaGetLastError();                                                                   \
            return gpcc::fail(1000 + (int)_e, std::string(#expr) + ": " + cudaGetErrorString(_e)); \
        }                                                                                         \
    } while (0)

template <class T>
struct DevBuf : DevArray<T> {   // growable device buffer (1.5x head-room) + pinned host mirror of the same size
    T* h = nullptr;
    ~DevBuf() { if (h) cudaFreeHost(h); }
    cudaError_t reserve(size_t n) {
        if (n <= this->cap) return cudaSuccess;
        if (h) cudaFreeHost(h);
        h = nullptr;
        size_t c = std::max<size_t>(n, 1024);
        c = c + c / 2;
        cudaError_t e = DevArray<T>::reserve(c);
        if (e != cudaSuccess) return e;
        e = cudaMallocHost(&h, c * sizeof(T));
        if (e != cudaSuccess) { h = nullptr; this->cap = 0; }   // no mirror: the next reserve allocates both again
        return e;
    }
};

// Staging of one evaluation batch (evaluate_on_device).
struct EvalSlot {
    DevBuf<double> delays, alpha, rho, ll, grad;
    DevBuf<int> info;
};

// Everything the context holds on one device.  Members are destroyed after the destructor's body, with `dev` current.
struct DeviceState {
    int dev = 0;
    Stream stream;
    EvalSlot slot;
    DevBuf<double> post_ll, post_prior, post_out;   // persistent staging of the posterior kernel (no cudaMalloc/cudaFree per call)
    // staging of the device-resident fit (small_fit.cu)
    DevBuf<double> fit_delays, fit_theta0, fit_ll, fit_theta;
    DevBuf<int> fit_iters, fit_nfev, fit_status, fit_order;
    DevBuf<unsigned long long> fit_counters;
    DevBuf<double> gat_send, gat_recv, gat_post;     // all-gather of the grid results (persistent: no cudaMalloc per call)
    Event ev0, ev1;                                  // around the small-N kernel launch of the call (profiling)
    LargeWorkspace large;     // tiled large-N path (large_path.cu)
    // per-call statistics (profiling)
    double ms_eval = 0, ms_assembly = 0, ms_factor = 0, ms_gradreduce = 0;
    long long launches = 0, evals = 0, evals_grad = 0, shared_prefix_evals = 0, tau_cache_evals = 0, assembly_bytes = 0;
    ~DeviceState() { cudaSetDevice(dev); }
};

struct SSSampleBuffers {
    DevArray<int> ints;                          // order, idx: [2 N]
    DevArray<double> step, aggA, aggc, f, z;     // SSSampleScratch; f [nsamples][N]; z [nsamples][N][d+1] (z_in, or the deviates)
};

struct FitStateDelete { void operator()(gpcc_fit_state* s) const { gpcc_fit_state_destroy(s); } };

}  // namespace gpcc

struct gpcc_ctx {
    std::vector<gpcc::DeviceState> ds;
    bool profiling = false;
    gpcc_stats stats{};
    gpcc::NcclBridge* nccl = nullptr;
    int world = 1, rank = 0;      // > 1 ranks: one process per device, joined by gpcc_ctx_comm_init_rank
};

struct gpcc_problem {
    gpcc_ctx* ctx = nullptr;
    int L = 0, N = 0, kernel_id = 0;
    std::vector<int> n_per_band, band, band_start;
    std::vector<double> t, y, sigma, mub, Sigmab, resid, s2, sigb;
    struct PerDev {
        int dev = 0;              // CUDA device id, copied from the context at creation: destroying a problem never reads the context
        gpcc::DevArray<double> t, resid, y, s2, sigb;
        gpcc::DevArray<int> band;
        gpcc::DevProblem dp;
        gpcc::DevArray<double> ss_t, ss_r, ss_s2;   // state-space method: each band sorted by t (gpcc_problem_set_method)
        gpcc::DevArray<int> ss_perm;                // ... and the input index of each of those points
        gpcc::SSSampleBuffers ss_smp;               // scratch and outputs of gpcc_ss_sample (first device), kept between calls
        gpcc::DevBuf<double> ss_postb;              // [L + L*L] postb of the filter
        gpcc::SSProblem ssp;
        ~PerDev() { cudaSetDevice(dev); }
    };
    std::vector<PerDev> pd;
    bool small_path = true;
    int method = GPCC_METHOD_DENSE;
    // fitted state of the last gpcc_postb / gpcc_predict* call (predict.cu); never handed to a caller
    std::unique_ptr<gpcc_fit_state, gpcc::FitStateDelete> cached_state;
};

namespace gpcc {
// Evaluate M (delay, alpha, rho) triples already staged in the pinned mirrors of ds[di].slot and wait for them;
// results land in ds[di].slot.ll.h / grad.h / info.h.
int evaluate_on_device(gpcc_problem* p, int di, int M, int want_grad);
int reserve_eval(gpcc_problem* p, int di, size_t M);
// postb of a GPCC_METHOD_STATESPACE problem: one filter on the first device
int statespace_postb(gpcc_problem* p, const double* delays, const double* alpha, double rho, double* out_mu, double* out_Sigma);
}  // namespace gpcc
