// Internal declarations shared by the CUDA translation units of libgpcc_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <algorithm>
#include <memory>
#include <string>
#include <type_traits>
#include <vector>

namespace gpcc {

constexpr int MAX_BANDS = 8;   // == GPCC_MAX_BANDS

// Device array that only ever grows, to exactly the size asked for (no cudaMalloc on repeated calls of the same size).
// It owns its memory and frees it when destroyed; the owner makes its device current first.
template <class T>
struct DevArray {
    T* d = nullptr;
    size_t cap = 0;
    DevArray() = default;
    DevArray(const DevArray&) = delete;
    DevArray& operator=(const DevArray&) = delete;
    ~DevArray() { if (d) cudaFree(d); }
    cudaError_t reserve(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (d) cudaFree(d);
        d = nullptr; cap = 0;
        cudaError_t e = cudaMalloc(&d, std::max<size_t>(n, 1) * sizeof(T));
        if (e == cudaSuccess) cap = n;
        else d = nullptr;
        return e;
    }
};

// Owning stream and event handles (cudaStream_t and cudaEvent_t are pointer types).
struct StreamDestroy { void operator()(cudaStream_t s) const { cudaStreamDestroy(s); } };
struct EventDestroy { void operator()(cudaEvent_t e) const { cudaEventDestroy(e); } };
using Stream = std::unique_ptr<std::remove_pointer_t<cudaStream_t>, StreamDestroy>;
using Event = std::unique_ptr<std::remove_pointer_t<cudaEvent_t>, EventDestroy>;
inline cudaError_t create_stream(Stream& s, int priority) {
    cudaStream_t h = nullptr;
    cudaError_t e = cudaStreamCreateWithPriority(&h, cudaStreamNonBlocking, priority);
    if (e == cudaSuccess) s.reset(h);
    return e;
}
inline cudaError_t create_event(Event& ev, unsigned flags = cudaEventDefault) {
    cudaEvent_t h = nullptr;
    cudaError_t e = cudaEventCreateWithFlags(&h, flags);
    if (e == cudaSuccess) ev.reset(h);
    return e;
}

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
struct LargeImpl;
struct LargeImplDelete { void operator()(LargeImpl* w) const; };
using LargeWorkspace = std::unique_ptr<LargeImpl, LargeImplDelete>;   // built on first use by large_eval
struct LargeTimings {
    double ms_assembly = 0, ms_factor = 0, ms_gradreduce = 0;
    long long launches = 0;
    long long shared_prefix_evals = 0;   // evaluations whose leading block was factorised by another matrix of their wave
    long long assembly_bytes = 0;        // HBM bytes moved by the covariance assembly kernels (tiles written; cache imports read + written)
    long long tau_cache_evals = 0;       // evaluations that imported the band-1 steps of their last band from the last-band cache
};
cudaError_t large_eval(const DevProblem& p, const EvalBatch& b, LargeWorkspace& ws, cudaStream_t stream, bool profile,
                       LargeTimings* timings);

// ---- state-space method for OU / matern32 / matern52 (statespace.cu): Kalman filter over the merged shifted times ----
struct SSProblem {
    int N = 0, L = 0;
    int band_start[MAX_BANDS + 1] = {0};
    double mub[MAX_BANDS] = {0}, Sigmab[MAX_BANDS] = {0};
    const double* t = nullptr;    // [N] each band sorted by t (stable argsort), bands concatenated
    const double* r = nullptr;    // [N] resid = y - mu_b in the same order
    const double* s2 = nullptr;   // [N] sigma^2 in the same order
};
// postb (may be NULL): with M = 1, receives the filter's final b-block, [L] mean + mu_b, then [L][L] covariance
cudaError_t statespace_launch(int kernel_id, const SSProblem& p, const EvalBatch& b, double* postb, cudaStream_t stream);
// Per merged training step k (N steps, D = d + L, NP = D (D+1) / 2), the moments behind the O(N) predictions of the state-space
// fit state: shifted time, band, filtered mean and packed covariance after the update, and the Bryson-Frazier adjoint of the
// step before its update (lam, Lam: smoothed mean m- - P- lam, smoothed covariance P- - P- Lam P-).
struct SSStore {
    double* t = nullptr;       // [N]
    int* band = nullptr;       // [N]
    double* m = nullptr;       // [N][D]
    double* P = nullptr;       // [N][NP]
    double* lam = nullptr;     // [N][D]
    double* Lam = nullptr;     // [N][NP]
};
// One forward filter that fills st (ll[0], info[0] as statespace_launch with M = 1), then the sequential backward pass (skipped
// when info[0] != 0).  hyp = [delays (L), alpha (L), rho] on the device.
cudaError_t statespace_store_launch(int kernel_id, const SSProblem& p, const double* hyp, double* ll, int* info,
                                    const SSStore& st, cudaStream_t stream);
// Smoothed predictive mean (+ mu_b) and standard deviation sqrt(max(var + 1e-8, 1e-6)) of NT test points (tt, band bt, any
// order) from st; p supplies N, L and the prior.  sd may be NULL.
cudaError_t statespace_predict_launch(int kernel_id, const SSProblem& p, const double* hyp, const SSStore& st, int NT,
                                      const double* tt, const int* bt, double* mu, double* sd, cudaStream_t stream);

// ---- exact O(N) draws of the state-space model (ss_sample.cu): the SDE recurrence over the merged times, as a scan ----
struct SSSampleArgs {
    double tau[MAX_BANDS] = {0}, alpha[MAX_BANDS] = {0}, rho = 0;
    unsigned long long seed = 0;
    int nsamples = 0;
    int sample0 = 0;              // generator counter of sample s: sample0 + s (a caller that draws in chunks of samples)
    unsigned tag = 0x53534D50u;   // generator stream: "SSMP" (gpcc_ss_sample), apart from the dense sampler's "GPCC" (predict.cu)
    const int* perm = nullptr;    // [N] input index of the point at each position of p's sorted per-band copy
    const double* zin = nullptr;  // [nsamples][N][d+1] deviates in input order, or NULL: Philox from (seed, sample, point)
    double* zout = nullptr;       // [nsamples][N][d+1] or NULL: the deviates used
    double* f = nullptr;          // [nsamples][N] draws in input order
};
struct SSSampleScratch {          // sizes from statespace_sample_scratch
    int* order = nullptr;         // [N] merged step -> sorted position
    int* idx = nullptr;           // [N] merged step -> input index
    double* step = nullptr;       // [N][d*d + d(d+1)/2 + 2] A, packed lower C, alpha, sigma of every merged step
    double* aggA = nullptr;       // [tiles][d*d]
    double* aggc = nullptr;       // [nsamples][tiles][d]
};
// doubles of SSSampleScratch::step, aggA and aggc (ints: 2 N)
void statespace_sample_scratch(int kernel_id, int N, int nsamples, size_t& n_step, size_t& n_aggA, size_t& n_aggc);
// Five launches on `stream`: merged ranks, per-step factors, tile aggregates, scan of the aggregates, tile re-run.
cudaError_t statespace_sample_launch(int kernel_id, const SSProblem& p, const SSSampleArgs& a, const SSSampleScratch& s,
                                     cudaStream_t stream);
// order[k] = the sorted position (in p) of merged step k: the filter's merge at delays tau (host, [L]).
cudaError_t statespace_rank_launch(const SSProblem& p, const double* tau, int* order, cudaStream_t stream);

// ---- exact O(N) posterior draws of the state-space fit state (ss_post_sample.cu): pathwise conditioning ----
// Doubles per merged training step of the records: A (d x d), gain k (D = d + L), 1 / S, alpha_l, residual.
int statespace_post_record_width(int kernel_id, int L);
// The records rec [N][width] and the input index in [N] of every merged training step, from the stored moments st of the fit
// state at hyp (device) / h_tau (host delays).  p: the training problem, each band sorted, on the device; perm: its input
// indices; order: [N] scratch.
cudaError_t statespace_post_records_launch(int kernel_id, const SSProblem& p, const double* hyp, const double* h_tau,
                                           const SSStore& st, const int* perm, int* order, double* rec, int* in,
                                           cudaStream_t stream);
// Per test point: tstep = the last training step at or before it (-1: none), tw [NT][2 D] = the weights c1, w of
// ss::point_mean_weights; need[step] |= 1 (a test point reads its m), 2 (... its adjoint).  need must be zeroed before.
cudaError_t statespace_post_locate_launch(int kernel_id, const SSProblem& p, const double* hyp, const SSStore& st, int NT,
                                          const double* tt, const int* bt, int* tstep, double* tw, int* need,
                                          cudaStream_t stream);
struct SSPostArgs {               // one chunk of C samples (global indices sample0 ..), all pointers on the device
    int N = 0, NT = 0, NM = 0, L = 0;    // training steps, test points, N + NT (the merged problem of the prior draw), bands
    int C = 0, sample0 = 0;
    unsigned long long seed = 0;
    unsigned tag = 0;                    // generator stream of the shift deviates (counter word 3 = 2)
    double mub[MAX_BANDS] = {0}, sqrt_sigmab[MAX_BANDS] = {0};
    const double* rec = nullptr;  const int* in = nullptr;     // records (statespace_post_records_launch)
    const int* band = nullptr;                                 // [N] band of every merged training step (SSStore::band)
    const int* tstep = nullptr;   const double* tw = nullptr;  const int* bt = nullptr;   // statespace_post_locate_launch
    const int* need = nullptr;
    int* mpos = nullptr;  int* lpos = nullptr;   // [N] slot of each flagged step (written by the chunk with sample0 = 0)
    const double* f = nullptr;    // [C][NM] prior draw of the merged problem, input order (training, then test points)
    const double* zin_b = nullptr;  double* zout_b = nullptr;  // [C][L] shift deviates in / out, or NULL
    double* bs = nullptr;         // [C][L] shift draws
    double* dv = nullptr;         // [N][C] pseudo-residuals, then innovations
    double* mbuf = nullptr;  double* lbuf = nullptr;          // [<= NT slots][D][C] m and lam~ at flagged steps
    double* out = nullptr;        // [C][NT] draws, test input order
};
// Shift draws, pseudo-residuals, forward and backward mean passes, test points: five launches on `stream`.
cudaError_t statespace_post_chunk_launch(int kernel_id, const SSPostArgs& a, cudaStream_t stream);

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
