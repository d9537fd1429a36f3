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
struct DevBuf {   // growable device buffer + pinned host mirror
    T* d = nullptr;
    T* h = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t n) {
        if (n <= cap) return cudaSuccess;
        release();
        size_t c = std::max<size_t>(n, 1024);
        c = c + c / 2;
        cudaError_t e = cudaMalloc(&d, c * sizeof(T));
        if (e != cudaSuccess) return e;
        e = cudaMallocHost(&h, c * sizeof(T));
        if (e != cudaSuccess) return e;
        cap = c;
        return cudaSuccess;
    }
    void release() {
        if (d) cudaFree(d);
        if (h) cudaFreeHost(h);
        d = nullptr; h = nullptr; cap = 0;
    }
};

// Staging of one evaluation batch (evaluate_on_device).
struct EvalSlot {
    DevBuf<double> delays, alpha, rho, ll, grad;
    DevBuf<int> info;
};

struct DeviceState {
    int dev = 0;
    cudaStream_t stream = nullptr;
    EvalSlot slot;
    DevBuf<double> post_ll, post_prior, post_out;   // persistent staging of the posterior kernel (no cudaMalloc/cudaFree per call)
    // staging of the device-resident fit (small_fit.cu)
    DevBuf<double> fit_delays, fit_theta0, fit_ll, fit_theta;
    DevBuf<int> fit_iters, fit_nfev, fit_status, fit_order;
    DevBuf<unsigned long long> fit_counters;
    DevBuf<double> gat_send, gat_recv, gat_post;     // all-gather of the grid results (persistent: no cudaMalloc per call)
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;        // around the small-N kernel launch of the call (profiling)
    LargeWorkspace large;     // tiled large-N path (large_path.cu)
    // per-call statistics (profiling)
    double ms_eval = 0, ms_assembly = 0, ms_factor = 0, ms_gradreduce = 0;
    long long launches = 0, evals = 0, evals_grad = 0, shared_prefix_evals = 0, tau_cache_evals = 0, assembly_bytes = 0;
};

}  // namespace gpcc

struct gpcc_ctx {
    std::vector<gpcc::DeviceState> ds;
    bool profiling = false;
    gpcc_stats stats{};
    gpcc::NcclBridge* nccl = nullptr;
    int world = 1, rank = 0;      // > 1 ranks: one process per device, joined by gpcc_ctx_comm_init_rank
};

struct gpcc_fit_state;

struct gpcc_problem {
    gpcc_ctx* ctx = nullptr;
    int L = 0, N = 0, kernel_id = 0;
    std::vector<int> n_per_band, band, band_start;
    std::vector<double> t, y, sigma, mub, Sigmab, resid, s2, sigb;
    struct PerDev {
        int dev = 0;              // CUDA device id, copied from the context at creation: destroying a problem never reads the context
        double *t = nullptr, *resid = nullptr, *y = nullptr, *s2 = nullptr, *sigb = nullptr;
        int* band = nullptr;
        gpcc::DevProblem dp;
    };
    std::vector<PerDev> pd;
    bool small_path = true;
    gpcc_fit_state* cached_state = nullptr;   // fitted state of the last gpcc_postb / gpcc_predict* call (predict.cu)
};

namespace gpcc {
// Evaluate M (delay, alpha, rho) triples already staged in the pinned mirrors of ds[di].slot and wait for them;
// results land in ds[di].slot.ll.h / grad.h / info.h.
int evaluate_on_device(gpcc_problem* p, int di, int M, int want_grad);
int reserve_eval(gpcc_problem* p, int di, size_t M);
}  // namespace gpcc
