// C ABI of libgpcc_b200.so (include/gpcc_b200.h): contexts, problems, batched evaluation, the
// host-driven batched L-BFGS fit, the grid posterior, postb and predictions.
// There is no CPU fallback anywhere in this file: every likelihood value comes from a CUDA kernel.
#include "state.h"
#include "lbfgs.h"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <memory>
#include <string>
#include <thread>
#include <utility>
#include <vector>

using namespace gpcc;

namespace gpcc {
namespace { thread_local std::string g_last_error; }
int fail(int code, const std::string& msg) {
    g_last_error = msg;
    return code;
}
const std::string& last_error() { return g_last_error; }
}  // namespace gpcc

namespace {

// ---- parameter transforms (gpccfixdelay_marginaliseb.jl:112-126; MiscUtil presumed) ---------------
inline double softplus(double x) { return x > 0 ? x + std::log1p(std::exp(-x)) : std::log1p(std::exp(x)); }
inline double logistic(double x) { return 0.5 * (1.0 + std::tanh(0.5 * x)); }

void unpack_theta(const double* theta, int L, const gpcc_fit_options& o, double* alpha, double* rho, double* jac) {
    for (int l = 0; l < L; ++l) {
        alpha[l] = softplus(theta[l]) + o.alpha_floor;                       // makeα (:112)
        if (jac) jac[l] = logistic(theta[l]);
    }
    const double s = logistic(theta[L]);
    *rho = o.rhomin + (o.rhomax - o.rhomin) * s;                             // makeρ (:114)
    if (jac) jac[L] = (o.rhomax - o.rhomin) * s * (1.0 - s);
}

int check_options(const gpcc_fit_options* o) {
    if (!o) return fail(-1, "options pointer is NULL");
    if (o->transform_id != GPCC_TRANSFORM_SOFTPLUS_LOGISTIC) return fail(-2, "unknown transform_id");
    if (!(o->rhomin > 0) || !(o->rhomax > o->rhomin)) return fail(-3, "need 0 < rhomin < rhomax");
    if (!(o->alpha_floor >= 0)) return fail(-4, "alpha_floor must be >= 0");
    if (o->optimizer != GPCC_OPT_LBFGS && o->optimizer != GPCC_OPT_NELDERMEAD) return fail(-5, "unknown optimizer");
    return 0;
}

}  // namespace
int gpcc::evaluate_on_device(gpcc_problem* p, int di, int M, int want_grad) {
    DeviceState& s = p->ctx->ds[di];
    EvalSlot& q = s.slot;
    const int L = p->L;
    CUDA_TRY(cudaSetDevice(s.dev));
    cudaStream_t stream = s.stream.get();
    CUDA_TRY(cudaMemcpyAsync(q.delays.d, q.delays.h, (size_t)M * L * sizeof(double), cudaMemcpyHostToDevice, stream));
    CUDA_TRY(cudaMemcpyAsync(q.alpha.d, q.alpha.h, (size_t)M * L * sizeof(double), cudaMemcpyHostToDevice, stream));
    CUDA_TRY(cudaMemcpyAsync(q.rho.d, q.rho.h, (size_t)M * sizeof(double), cudaMemcpyHostToDevice, stream));
    EvalBatch b;
    b.M = M; b.delays = q.delays.d; b.alpha = q.alpha.d; b.rho = q.rho.d; b.want_grad = want_grad;
    b.ll = q.ll.d; b.grad = q.grad.d; b.info = q.info.d;
    b.h_delays = q.delays.h; b.h_alpha = q.alpha.h; b.h_rho = q.rho.h;
    const bool prof = p->ctx->profiling;
    const bool one_kernel = p->method == GPCC_METHOD_STATESPACE || p->small_path;
    if (one_kernel) {
        if (prof) CUDA_TRY(cudaEventRecord(s.ev0.get(), stream));
        if (p->method == GPCC_METHOD_STATESPACE) CUDA_TRY(statespace_launch(p->kernel_id, p->pd[di].ssp, b, nullptr, stream));
        else CUDA_TRY(small_sweep_launch(p->pd[di].dp, b, stream));
        if (prof) CUDA_TRY(cudaEventRecord(s.ev1.get(), stream));
        s.launches += 1;
    } else {
        LargeTimings lt;
        CUDA_TRY(large_eval(p->pd[di].dp, b, s.large, stream, prof, &lt));
        s.launches += lt.launches;
        s.ms_assembly += lt.ms_assembly; s.ms_factor += lt.ms_factor; s.ms_gradreduce += lt.ms_gradreduce;
        s.ms_eval += lt.ms_assembly + lt.ms_factor + lt.ms_gradreduce;
        s.shared_prefix_evals += lt.shared_prefix_evals;
        s.tau_cache_evals += lt.tau_cache_evals;
        s.assembly_bytes += lt.assembly_bytes;
    }
    CUDA_TRY(cudaMemcpyAsync(q.ll.h, q.ll.d, (size_t)M * sizeof(double), cudaMemcpyDeviceToHost, stream));
    if (want_grad)
        CUDA_TRY(cudaMemcpyAsync(q.grad.h, q.grad.d, (size_t)M * (L + 1) * sizeof(double), cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(cudaMemcpyAsync(q.info.h, q.info.d, (size_t)M * sizeof(int), cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(cudaStreamSynchronize(stream));
    if (prof && one_kernel) {
        float ms = 0;
        CUDA_TRY(cudaEventElapsedTime(&ms, s.ev0.get(), s.ev1.get()));
        s.ms_eval += ms;
    }
    s.evals += M;
    if (want_grad) s.evals_grad += M;
    return 0;
}

int gpcc::reserve_eval(gpcc_problem* p, int di, size_t M) {
    DeviceState& s = p->ctx->ds[di];
    EvalSlot& q = s.slot;
    const int L = p->L;
    CUDA_TRY(cudaSetDevice(s.dev));
    CUDA_TRY(q.delays.reserve(M * L));
    CUDA_TRY(q.alpha.reserve(M * L));
    CUDA_TRY(q.rho.reserve(M));
    CUDA_TRY(q.ll.reserve(M));
    CUDA_TRY(q.grad.reserve(M * (L + 1)));
    CUDA_TRY(q.info.reserve(M));
    return 0;
}

namespace {
void reset_stats(gpcc_ctx* ctx) {
    for (auto& s : ctx->ds) {
        s.ms_eval = s.ms_assembly = s.ms_factor = s.ms_gradreduce = 0;
        s.launches = s.evals = s.evals_grad = s.shared_prefix_evals = s.tau_cache_evals = s.assembly_bytes = 0;
        // the call about to start refills the pinned staging buffers: wait for what may still read them (a call that
        // failed midway, or the all-gather of posterior_on_devices, which synchronises device 0 only)
        cudaSetDevice(s.dev);
        cudaStreamSynchronize(s.stream.get());
    }
}

void collect_stats(gpcc_ctx* ctx, const gpcc_problem* p, double ms_total) {
    gpcc_stats st{};
    st.ms_total = ms_total;
    for (auto& s : ctx->ds) {
        st.ms_eval_kernels = std::max(st.ms_eval_kernels, s.ms_eval);   // devices run concurrently
        st.ms_assembly = std::max(st.ms_assembly, s.ms_assembly);
        st.ms_factor = std::max(st.ms_factor, s.ms_factor);
        st.ms_gradreduce = std::max(st.ms_gradreduce, s.ms_gradreduce);
        st.n_eval_launches += s.launches;
        st.n_evals += s.evals;
        st.n_evals_grad += s.evals_grad;
        st.n_shared_prefix += s.shared_prefix_evals;
        st.n_tau_cache += s.tau_cache_evals;
        st.assembly_bytes = std::max(st.assembly_bytes, s.assembly_bytes);   // like ms_assembly: the busiest device
    }
    st.path = !p ? 0 : p->method == GPCC_METHOD_STATESPACE ? 2 : p->small_path ? 0 : 1;
    st.n_devices = (int)ctx->ds.size();
    ctx->stats = st;
}

// total order on doubles by bit pattern (NaN-safe: the sort keys below may contain invalid hyper-parameters)
inline bool bits_less(double a, double b, bool& decided) {
    unsigned long long x, y;
    std::memcpy(&x, &a, 8); std::memcpy(&y, &b, 8);
    decided = x != y;
    return x < y;
}

struct Timer {
    std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
    double ms() const { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(); }
};

// ---- the fit of one device's shard ------------------------------------------------------------------
struct FitOutputs {
    double *ll, *theta, *alpha, *rho;
    int *iters, *nfev, *info;
};

void write_fit_outputs(const gpcc_problem* p, const gpcc_fit_options& o, const FitOutputs& out, int gi, double f, const double* x,
                       int iters, int nfev, int status) {
    const int L = p->L, n = L + 1;
    if (out.ll) out.ll[gi] = -f;                                           // -result.minimum (:351)
    if (out.iters) out.iters[gi] = iters;
    if (out.nfev) out.nfev[gi] = nfev;
    if (out.info) out.info[gi] = status;
    double a_[LBFGS_MAXN], r_ = std::numeric_limits<double>::quiet_NaN();
    if (status == LbfgsState::NO_START) {
        for (int k = 0; k < L; ++k) a_[k] = std::numeric_limits<double>::quiet_NaN();
        if (out.theta) for (int k = 0; k < n; ++k) out.theta[(size_t)gi * n + k] = std::numeric_limits<double>::quiet_NaN();
    } else {
        unpack_theta(x, L, o, a_, &r_, nullptr);                            // unpack(paramopt) (:235)
        if (out.theta) std::memcpy(out.theta + (size_t)gi * n, x, n * sizeof(double));
    }
    if (out.alpha) std::memcpy(out.alpha + (size_t)gi * L, a_, L * sizeof(double));
    if (out.rho) out.rho[gi] = r_;
}

// Fused small-N path: the whole shard in ONE launch of the persistent fit kernel (small_fit.cu) -- screening, L-BFGS and
// every likelihood / gradient evaluation stay on the device; the host uploads delays + start points and reads the optima.
int fit_shard_device(gpcc_problem* p, int di, const std::vector<int>& idx, const double* delays, int P, const double* theta0,
                     const gpcc_fit_options& o, const FitOutputs& out) {
    const int L = p->L, n = L + 1;
    const int m = (int)idx.size();
    DeviceState& s = p->ctx->ds[di];
    CUDA_TRY(cudaSetDevice(s.dev));
    const size_t nth = (size_t)(o.theta0_per_candidate ? m : 1) * P * n;
    CUDA_TRY(s.fit_delays.reserve((size_t)m * L));
    CUDA_TRY(s.fit_theta0.reserve(nth));
    CUDA_TRY(s.fit_ll.reserve(m));
    CUDA_TRY(s.fit_theta.reserve((size_t)m * n));
    CUDA_TRY(s.fit_iters.reserve(m));
    CUDA_TRY(s.fit_nfev.reserve(m));
    CUDA_TRY(s.fit_status.reserve(m));
    CUDA_TRY(s.fit_counters.reserve(8));
    CUDA_TRY(s.fit_order.reserve(m));
    for (int c = 0; c < m; ++c) std::memcpy(s.fit_delays.h + (size_t)c * L, delays + (size_t)idx[c] * L, L * sizeof(double));
    if (o.theta0_per_candidate)
        for (int c = 0; c < m; ++c) std::memcpy(s.fit_theta0.h + (size_t)c * P * n, theta0 + (size_t)idx[c] * P * n, (size_t)P * n * sizeof(double));
    else
        std::memcpy(s.fit_theta0.h, theta0, (size_t)P * n * sizeof(double));
    // Work-queue order.  A persistent CTA runs its candidate to convergence, so the launch ends when the last-started long
    // candidate ends: candidates that are likely to need many iterations should start first.  Evaluation counts are hardly
    // predictable (measured: correlation 0.2 with the screening likelihood or with the neighbours on the grid), except that
    // the flattest likelihoods -- and with them the longest L-BFGS runs -- sit where the light curves overlap least, i.e. at
    // the largest spread of delays (profiles/README.md, scheduling study: grid order 13 % over the ideal span, this 5 %).
    // The order cannot change any result: candidates never interact.
    {
        std::vector<std::pair<double, int>> key(m);
        for (int c = 0; c < m; ++c) {
            const double* dl = delays + (size_t)idx[c] * L;
            double lo = dl[0], hi = dl[0];
            for (int l = 1; l < L; ++l) { lo = std::min(lo, dl[l]); hi = std::max(hi, dl[l]); }
            key[c] = {-(hi - lo), c};
        }
        std::stable_sort(key.begin(), key.end(), [](const std::pair<double, int>& a, const std::pair<double, int>& b) { return a.first < b.first; });
        for (int c = 0; c < m; ++c) s.fit_order.h[c] = key[c].second;
    }
    for (int k = 0; k < 8; ++k) s.fit_counters.h[k] = 0;
    s.fit_counters.h[5] = ~0ULL;
    cudaStream_t st = s.stream.get();
    CUDA_TRY(cudaMemcpyAsync(s.fit_delays.d, s.fit_delays.h, (size_t)m * L * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(s.fit_theta0.d, s.fit_theta0.h, nth * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(s.fit_counters.d, s.fit_counters.h, 8 * sizeof(unsigned long long), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(s.fit_order.d, s.fit_order.h, (size_t)m * sizeof(int), cudaMemcpyHostToDevice, st));
    FitParams fp;
    fp.M = m; fp.P = P; fp.theta0_per_candidate = o.theta0_per_candidate; fp.max_iter = o.max_iter;
    fp.rhomin = o.rhomin; fp.rhomax = o.rhomax; fp.alpha_floor = o.alpha_floor; fp.gtol = o.gtol; fp.ftol = o.ftol;
    fp.history = o.history;
    fp.optimizer = o.optimizer; fp.nm_gtol = o.nm_gtol;
    FitBuffers fb;
    fb.delays = s.fit_delays.d; fb.theta0 = s.fit_theta0.d; fb.ll = s.fit_ll.d; fb.theta = s.fit_theta.d;
    fb.iters = s.fit_iters.d; fb.nfev = s.fit_nfev.d; fb.status = s.fit_status.d; fb.counters = s.fit_counters.d;
    fb.order = s.fit_order.d;
    const bool prof = p->ctx->profiling;
    if (prof) CUDA_TRY(cudaEventRecord(s.ev0.get(), st));
    CUDA_TRY(small_fit_launch(p->pd[di].dp, fp, fb, st));
    if (prof) CUDA_TRY(cudaEventRecord(s.ev1.get(), st));
    CUDA_TRY(cudaMemcpyAsync(s.fit_ll.h, s.fit_ll.d, (size_t)m * sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(s.fit_theta.h, s.fit_theta.d, (size_t)m * n * sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(s.fit_iters.h, s.fit_iters.d, (size_t)m * sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(s.fit_nfev.h, s.fit_nfev.d, (size_t)m * sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(s.fit_status.h, s.fit_status.d, (size_t)m * sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(s.fit_counters.h, s.fit_counters.d, 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (prof) {
        float ms = 0;
        CUDA_TRY(cudaEventElapsedTime(&ms, s.ev0.get(), s.ev1.get()));
        s.ms_eval += ms;
    }
    static const bool debug = getenv("GPCC_FIT_DEBUG") != nullptr;
    if (debug && s.fit_counters.h[6] > 0) {
        const double span = (double)(s.fit_counters.h[4] - s.fit_counters.h[5]) * 1e-6;
        const double mean_exit = (double)s.fit_counters.h[3] / (double)s.fit_counters.h[6] * 1e-6;
        fprintf(stderr, "[gpcc fit] %d candidates on %llu CTAs: kernel span %.2f ms, mean CTA exit at %.2f ms (%.1f %% of the CTA-time busy), "
                        "%llu gradient + %llu forward evaluations\n", m, s.fit_counters.h[6], span, mean_exit, 100.0 * mean_exit / span,
                s.fit_counters.h[1], s.fit_counters.h[2]);
        if (s.fit_counters.h[7])
            fprintf(stderr, "[gpcc fit] thread-0 optimiser time: %.1f cycles per evaluation (build with -DGPCC_FIT_PROF)\n",
                    (double)s.fit_counters.h[7] / (double)(s.fit_counters.h[1] + s.fit_counters.h[2]));
    }
    s.launches += 1;
    s.evals += (long long)(s.fit_counters.h[1] + s.fit_counters.h[2]);
    s.evals_grad += (long long)s.fit_counters.h[1];
    for (int c = 0; c < m; ++c)
        write_fit_outputs(p, o, out, idx[c], -s.fit_ll.h[c], s.fit_theta.h + (size_t)c * n, s.fit_iters.h[c], s.fit_nfev.h[c], s.fit_status.h[c]);
    return 0;
}

// Candidates idx[0..n) (global indices) are fitted on device `di`.  The host-driven batched L-BFGS below is the driver of
// the tiled path; on the fused small-N path it runs only under GPCC_FIT_HOST=1, as the reference that the persistent fit
// kernel is tested against.
int fit_shard(gpcc_problem* p, int di, const std::vector<int>& idx, const double* delays, int P, const double* theta0,
              const gpcc_fit_options& o, const FitOutputs& out) {
    const int L = p->L, n = L + 1;
    const int m = (int)idx.size();
    if (m == 0) return 0;
    static const bool host_loop = getenv("GPCC_FIT_HOST") != nullptr;
    const bool dense = p->method == GPCC_METHOD_DENSE;
    if (dense && p->small_path && (!host_loop || o.optimizer == GPCC_OPT_NELDERMEAD))
        return fit_shard_device(p, di, idx, delays, P, theta0, o, out);
    if (o.optimizer == GPCC_OPT_NELDERMEAD)
        return fail(-7, dense ? "the Nelder-Mead option runs on the fused small-N path only (N <= 199); use the default L-BFGS"
                              : "the Nelder-Mead option runs on the fused small-N dense path only; use the default L-BFGS");
    EvalSlot& q = p->ctx->ds[di].slot;
    LbfgsOptions lo;
    lo.max_iter = o.max_iter; lo.gtol = o.gtol; lo.ftol = o.ftol; lo.history = o.history; lo.n_scale = L;

    std::vector<LbfgsState> st(m);
    std::vector<double> jac(n);
    // ---- stage 1: screening of the P start points (:207-209), batched over all candidates -----------
    const int screen_grad = o.max_iter > 0 ? 1 : 0;      // iterations = 0: the fixed-theta sweep, forward-only evaluations
    // chunked so that one batch never exceeds ~1M evaluations worth of staging
    const size_t chunk_c = std::max<size_t>(1, std::min<size_t>(m, (size_t)(1 << 18) / std::max(1, P)));
    int rc = reserve_eval(p, di, chunk_c * P);
    if (rc) return rc;
    std::vector<int> seq(m);
    for (int c = 0; c < m; ++c) seq[c] = c;
    if (dense && !p->small_path && o.max_iter <= 0 && !o.theta0_per_candidate && L >= 2) {
        // fixed-theta sweep on the tiled path (forward-only evaluations): candidates that share the delays of all bands but
        // the last become neighbours, so that a wave factorises their common leading block once (large_path.cu)
        std::stable_sort(seq.begin(), seq.end(), [&](int x, int y) {
            const double* dx = delays + (size_t)idx[x] * L;
            const double* dy = delays + (size_t)idx[y] * L;
            bool dec;
            for (int l = 0; l + 1 < L; ++l) { const bool lt = bits_less(dx[l], dy[l], dec); if (dec) return lt; }
            return false;
        });
    }
    for (size_t c0 = 0; c0 < (size_t)m; c0 += chunk_c) {
        const int* cand = seq.data() + c0;
        const size_t nc = std::min<size_t>(m, c0 + chunk_c) - c0;
        for (size_t a = 0; a < nc; ++a) {              // evaluations cand-major, P per candidate
            const int gi = idx[cand[a]];
            for (int j = 0; j < P; ++j) {
                const size_t e = a * P + j;
                const double* th = o.theta0_per_candidate ? theta0 + ((size_t)gi * P + j) * n : theta0 + (size_t)j * n;
                std::memcpy(q.delays.h + e * L, delays + (size_t)gi * L, L * sizeof(double));
                unpack_theta(th, L, o, q.alpha.h + e * L, q.rho.h + e, nullptr);
            }
        }
        rc = evaluate_on_device(p, di, (int)(nc * P), screen_grad);
        if (rc) return rc;
        for (size_t a = 0; a < nc; ++a) {
            const int c = cand[a], gi = idx[c];
            int best = -1;
            double bestf = std::numeric_limits<double>::infinity();
            for (int j = 0; j < P; ++j) {          // argmin of -logL, first minimum wins (Julia argmin, :209)
                const size_t e = a * P + j;
                const double f = -q.ll.h[e];
                if (q.info.h[e] == 0 && std::isfinite(f) && f < bestf) { bestf = f; best = j; }
            }
            LbfgsState& S = st[c];
            S.n = n;
            S.nfev = P;
            if (best < 0) { S.status = LbfgsState::NO_START; S.f = std::numeric_limits<double>::infinity(); continue; }
            const size_t e = a * P + best;
            const double* th = o.theta0_per_candidate ? theta0 + ((size_t)gi * P + best) * n : theta0 + (size_t)best * n;
            if (o.max_iter <= 0) {           // screening only (:207-209): the evaluations ran without gradient
                lb_copy(S.x, th, n);
                S.f = bestf; S.iters = 0; S.status = LbfgsState::ITER_CAP;
                continue;
            }
            double a_[LBFGS_MAXN], r_, g_[LBFGS_MAXN];
            unpack_theta(th, L, o, a_, &r_, jac.data());
            for (int k = 0; k < n; ++k) g_[k] = -q.grad.h[e * n + k] * jac[k];
            S.start(n, th, bestf, g_, lo);
        }
    }
    // ---- stage 2: batched L-BFGS, one evaluation of every running candidate per round -----------------------
    std::vector<int> active;
    for (int c = 0; c < m; ++c)
        if (st[c].status == LbfgsState::RUNNING) active.push_back(c);
    rc = reserve_eval(p, di, active.size());
    if (rc) return rc;
    while (!active.empty()) {
        const int na = (int)active.size();
        for (int a = 0; a < na; ++a) {
            const int c = active[a];
            std::memcpy(q.delays.h + (size_t)a * L, delays + (size_t)idx[c] * L, L * sizeof(double));
            unpack_theta(st[c].xt, L, o, q.alpha.h + (size_t)a * L, q.rho.h + a, nullptr);
        }
        rc = evaluate_on_device(p, di, na, 1);
        if (rc) return rc;
        size_t w = 0;
        for (int a = 0; a < na; ++a) {
            const int c = active[a];
            LbfgsState& S = st[c];
            double a_[LBFGS_MAXN], r_, g_[LBFGS_MAXN];
            unpack_theta(S.xt, L, o, a_, &r_, jac.data());
            const bool ok = q.info.h[a] == 0 && std::isfinite(q.ll.h[a]);
            for (int k = 0; k < n; ++k) g_[k] = ok ? -q.grad.h[(size_t)a * n + k] * jac[k] : 0.0;
            S.feed(ok, -q.ll.h[a], g_, lo);
            if (S.status == LbfgsState::RUNNING) active[w++] = c;
        }
        active.resize(w);
    }
    // ---- outputs ------------------------------------------------------------------------------------------
    for (int c = 0; c < m; ++c) write_fit_outputs(p, o, out, idx[c], st[c].f, st[c].x, st[c].iters, st[c].nfev, st[c].status);
    return 0;
}

// Run fn(di) on every device of the context concurrently (one host thread per device).
template <class F>
int for_each_device(gpcc_ctx* ctx, F fn) {
    const int nd = (int)ctx->ds.size();
    if (nd == 1) return fn(0);
    std::vector<int> rcs(nd, 0);
    std::vector<std::string> errs(nd);
    std::vector<std::thread> th;
    for (int di = 0; di < nd; ++di)
        th.emplace_back([&, di]() { rcs[di] = fn(di); errs[di] = gpcc::last_error(); });
    for (auto& t : th) t.join();
    for (int di = 0; di < nd; ++di)
        if (rcs[di]) return fail(rcs[di], "device " + std::to_string(ctx->ds[di].dev) + ": " + errs[di]);
    return 0;
}

int fit_all(gpcc_problem* p, int M, const double* delays, int P, const double* theta0, const gpcc_fit_options& o,
            const FitOutputs& out) {
    gpcc_ctx* ctx = p->ctx;
    const int nd = (int)ctx->ds.size();
    std::vector<std::vector<int>> shard(nd);
    // candidate m -> global device m mod G (SURVEY 8e), G = ranks x devices per rank; this process owns G-indices rank*nd + di
    const int G = ctx->world * nd;
    for (int m = 0; m < M; ++m) {
        const int g = m % G;
        if (g / nd == ctx->rank) shard[g % nd].push_back(m);
    }
    return for_each_device(ctx, [&](int di) { return fit_shard(p, di, shard[di], delays, P, theta0, o, out); });
}

}  // namespace

// =====================================================================================================
extern "C" {

int gpcc_version(void) { return 103; }   // 103: gpcc_ss_state_*, then gpcc_ss_sample and gpcc_ss_state_sample (additive, same number); 102: gpcc_problem_set_method; 101: gpcc_stats grew by n_tau_cache and assembly_bytes
const char* gpcc_last_error(void) { return gpcc::last_error().c_str(); }

int gpcc_fit_options_default(gpcc_fit_options* o) {
    if (!o) return fail(-1, "options pointer is NULL");
    o->max_iter = 1000;
    o->rhomin = 0.1;
    o->rhomax = 20.0;
    o->alpha_floor = 1e-8;
    o->gtol = 1e-7;
    o->ftol = 1e-13;
    o->history = 8;
    o->transform_id = GPCC_TRANSFORM_SOFTPLUS_LOGISTIC;
    o->theta0_per_candidate = 0;
    o->optimizer = GPCC_OPT_LBFGS;
    o->nm_gtol = 1e-6;
    return 0;
}

int gpcc_ctx_create(int ndev, const int* dev_ids, gpcc_ctx** out) {
    if (!out) return fail(-1, "out is NULL");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        cudaGetLastError();
        return fail(1000 + (int)e, std::string("no CUDA device available (this library has no CPU fallback): ") +
                                       cudaGetErrorString(e));
    }
    if (ndev <= 0) ndev = 1;
    if (ndev > count) return fail(-2, "ndev exceeds the number of visible CUDA devices");
    // every id is checked before a DeviceState holds it: its destructor makes its device current
    std::vector<int> devs(ndev);
    for (int i = 0; i < ndev; ++i) {
        devs[i] = dev_ids ? dev_ids[i] : i;
        if (devs[i] < 0 || devs[i] >= count) return fail(-3, "invalid device id");
        cudaDeviceProp prop;
        CUDA_TRY(cudaGetDeviceProperties(&prop, devs[i]));
        if (prop.major < 10) return fail(-4, "libgpcc_b200 is built for sm_100a (Blackwell B200) only");
    }
    std::unique_ptr<gpcc_ctx> ctx(new gpcc_ctx());
    ctx->ds = std::vector<DeviceState>(ndev);     // DeviceState owns device resources: not movable, so no resize()
    for (int i = 0; i < ndev; ++i) ctx->ds[i].dev = devs[i];
    for (DeviceState& s : ctx->ds) {
        CUDA_TRY(cudaSetDevice(s.dev));
        // highest priority: in the tiled path this stream carries the critical pivot/panel chain while the bulk of each
        // trailing update runs on a low-priority stream (large_path.cu), so pivot CTAs get the next free SM
        int prio_lo = 0, prio_hi = 0;
        CUDA_TRY(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
        CUDA_TRY(create_stream(s.stream, prio_hi));
        CUDA_TRY(create_event(s.ev0));
        CUDA_TRY(create_event(s.ev1));
    }
    *out = ctx.release();
    return 0;
}

int gpcc_ctx_destroy(gpcc_ctx* ctx) {
    if (!ctx) return 0;
    if (ctx->nccl) nccl_bridge_destroy(ctx->nccl);
    delete ctx;
    return 0;
}

int gpcc_ctx_set_profiling(gpcc_ctx* ctx, int enabled) {
    if (!ctx) return fail(-1, "ctx is NULL");
    ctx->profiling = enabled != 0;
    return 0;
}
int gpcc_ctx_get_stats(const gpcc_ctx* ctx, gpcc_stats* out) {
    if (!ctx || !out) return fail(-1, "NULL argument");
    *out = ctx->stats;
    return 0;
}
int gpcc_ctx_device_count(const gpcc_ctx* ctx) { return ctx ? (int)ctx->ds.size() : 0; }

int gpcc_problem_create(gpcc_ctx* ctx, int L, const int* n_per_band, const double* t, const double* y,
                        const double* sigma, int kernel_id, const double* mub, const double* Sigmab,
                        gpcc_problem** out) {
    if (!ctx || !out || !n_per_band || !t || !y || !sigma) return fail(-1, "NULL argument");
    *out = nullptr;
    if (L < 1 || L > GPCC_MAX_BANDS) return fail(-2, "L must be in 1..GPCC_MAX_BANDS");
    if (kernel_id < 0 || kernel_id > 3)
        return fail(-3, "unknown kernel (expected GPCC.OU, GPCC.rbf, GPCC.matern32 or GPCC.matern52)");
    std::unique_ptr<gpcc_problem> p(new gpcc_problem());
    p->ctx = ctx; p->L = L; p->kernel_id = kernel_id;
    p->n_per_band.assign(n_per_band, n_per_band + L);
    p->band_start.assign(L + 1, 0);
    for (int l = 0; l < L; ++l) {
        if (n_per_band[l] < 1) return fail(-4, "every band needs at least one observation");
        p->band_start[l + 1] = p->band_start[l] + n_per_band[l];
    }
    const int N = p->N = p->band_start[L];
    p->t.assign(t, t + N); p->y.assign(y, y + N); p->sigma.assign(sigma, sigma + N);
    p->mub.resize(L); p->Sigmab.resize(L);
    for (int l = 0; l < L; ++l) {
        const int a = p->band_start[l], b = p->band_start[l + 1], n = b - a;
        if (mub) p->mub[l] = mub[l];
        else {                                           // mean(y_l)   (gpccfixdelay_marginaliseb.jl:92)
            double s = 0; for (int i = a; i < b; ++i) s += y[i];
            p->mub[l] = s / n;
        }
        if (Sigmab) p->Sigmab[l] = Sigmab[l];
        else {                                           // 100*var(y_l), unbiased (:94)
            double s = 0; for (int i = a; i < b; ++i) s += y[i];
            const double mean = s / n;
            double v = 0; for (int i = a; i < b; ++i) v += (y[i] - mean) * (y[i] - mean);
            p->Sigmab[l] = n > 1 ? 100.0 * v / (n - 1) : std::numeric_limits<double>::quiet_NaN();
        }
        if (!(p->Sigmab[l] > 0) || !std::isfinite(p->mub[l]))
            return fail(-5, "prior of the shift b is degenerate (band with <2 points or zero variance)");
    }
    p->band.resize(N); p->resid.resize(N); p->s2.resize(N); p->sigb.resize(N);
    for (int l = 0; l < L; ++l)
        for (int i = p->band_start[l]; i < p->band_start[l + 1]; ++i) {
            p->band[i] = l;
            p->resid[i] = y[i] - p->mub[l];              // Y - Q*mu_b (:98, :139)
            p->s2[i] = sigma[i] * sigma[i];              // Sobs (:89)
            p->sigb[i] = p->Sigmab[l];                   // B = Q Sigma_b Q' (:96)
            if (!std::isfinite(t[i]) || !std::isfinite(y[i]) || !std::isfinite(sigma[i]))
                return fail(-6, "non-finite input data");
        }
    p->small_path = small_path_supports(N);
    p->pd = std::vector<gpcc_problem::PerDev>(ctx->ds.size());   // not movable, like DeviceState
    for (size_t di = 0; di < ctx->ds.size(); ++di) p->pd[di].dev = ctx->ds[di].dev;   // before a failed upload destroys them
    for (auto& d : p->pd) {
        CUDA_TRY(cudaSetDevice(d.dev));
        CUDA_TRY(d.t.reserve(N));
        CUDA_TRY(d.resid.reserve(N));
        CUDA_TRY(d.y.reserve(N));
        CUDA_TRY(d.s2.reserve(N));
        CUDA_TRY(d.sigb.reserve(N));
        CUDA_TRY(d.band.reserve(N));
        CUDA_TRY(cudaMemcpy(d.t.d, p->t.data(), N * sizeof(double), cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMemcpy(d.resid.d, p->resid.data(), N * sizeof(double), cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMemcpy(d.y.d, p->y.data(), N * sizeof(double), cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMemcpy(d.s2.d, p->s2.data(), N * sizeof(double), cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMemcpy(d.sigb.d, p->sigb.data(), N * sizeof(double), cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMemcpy(d.band.d, p->band.data(), N * sizeof(int), cudaMemcpyHostToDevice));
        d.dp.N = N; d.dp.L = L; d.dp.kernel_id = kernel_id;
        d.dp.t = d.t.d; d.dp.resid = d.resid.d; d.dp.y = d.y.d; d.dp.s2 = d.s2.d; d.dp.sigb = d.sigb.d; d.dp.band = d.band.d;
        for (int l = 0; l <= L; ++l) d.dp.band_start[l] = p->band_start[l];
    }
    *out = p.release();
    return 0;
}

int gpcc_problem_destroy(gpcc_problem* p) {
    // only the problem's own copies of the device ids are read here (PerDev::dev): the context may already be gone
    // (finalizer order in Julia / Python is unspecified), see the lifetime rule in include/gpcc_b200.h
    delete p;
    return 0;
}

int gpcc_problem_get_prior(const gpcc_problem* p, double* mub, double* Sigmab) {
    if (!p) return fail(-1, "problem is NULL");
    if (mub) std::memcpy(mub, p->mub.data(), p->L * sizeof(double));
    if (Sigmab) std::memcpy(Sigmab, p->Sigmab.data(), p->L * sizeof(double));
    return 0;
}

}  // extern "C"

// Per band, a stable argsort of t: the merge of the filter (statespace.cu) keeps this order within a band.  ord (may be
// NULL) receives the input index of every sorted point.
static void sort_bands(const gpcc_problem* p, std::vector<double>& t, std::vector<double>& r, std::vector<double>& s2,
                       std::vector<int>* ord_out = nullptr) {
    const int N = p->N;
    std::vector<int> ord(N);
    for (int i = 0; i < N; ++i) ord[i] = i;
    for (int l = 0; l < p->L; ++l)
        std::stable_sort(ord.begin() + p->band_start[l], ord.begin() + p->band_start[l + 1],
                         [&](int a, int b) { return p->t[a] < p->t[b]; });
    t.resize(N); r.resize(N); s2.resize(N);
    for (int i = 0; i < N; ++i) { t[i] = p->t[ord[i]]; r[i] = p->resid[ord[i]]; s2[i] = p->s2[ord[i]]; }
    if (ord_out) ord_out->swap(ord);
}

extern "C" {

int gpcc_problem_set_method(gpcc_problem* p, int method) {
    if (!p) return fail(-1, "problem is NULL");
    if (method != GPCC_METHOD_DENSE && method != GPCC_METHOD_STATESPACE) return fail(-2, "unknown method");
    if (method == GPCC_METHOD_STATESPACE && p->kernel_id == GPCC_KERNEL_RBF)
        return fail(-3, "the state-space method needs a Markovian kernel (OU, matern32 or matern52): rbf has no finite state-space form");
    if (method == GPCC_METHOD_STATESPACE) {
        const int N = p->N, L = p->L;
        std::vector<double> t, r, s2;
        std::vector<int> ord;
        sort_bands(p, t, r, s2, &ord);
        for (auto& d : p->pd) {
            CUDA_TRY(cudaSetDevice(d.dev));
            CUDA_TRY(d.ss_t.reserve(N));
            CUDA_TRY(d.ss_r.reserve(N));
            CUDA_TRY(d.ss_s2.reserve(N));
            CUDA_TRY(d.ss_perm.reserve(N));
            CUDA_TRY(d.ss_postb.reserve((size_t)L + (size_t)L * L));
            CUDA_TRY(cudaMemcpy(d.ss_t.d, t.data(), N * sizeof(double), cudaMemcpyHostToDevice));
            CUDA_TRY(cudaMemcpy(d.ss_r.d, r.data(), N * sizeof(double), cudaMemcpyHostToDevice));
            CUDA_TRY(cudaMemcpy(d.ss_s2.d, s2.data(), N * sizeof(double), cudaMemcpyHostToDevice));
            CUDA_TRY(cudaMemcpy(d.ss_perm.d, ord.data(), N * sizeof(int), cudaMemcpyHostToDevice));
            SSProblem& q = d.ssp;
            q.N = N; q.L = L;
            for (int l = 0; l <= L; ++l) q.band_start[l] = p->band_start[l];
            for (int l = 0; l < L; ++l) { q.mub[l] = p->mub[l]; q.Sigmab[l] = p->Sigmab[l]; }
            q.t = d.ss_t.d; q.r = d.ss_r.d; q.s2 = d.ss_s2.d;
        }
    }
    p->method = method;
    return 0;
}

static int loglik_batch_impl(gpcc_problem* p, int M, const double* delays, const double* alpha, const double* rho,
                             const double* theta, const gpcc_fit_options* o, int want_grad, double* out_ll,
                             double* out_grad, int* out_info) {
    if (!p || !delays || !out_ll) return fail(-1, "NULL argument");
    if (M < 0) return fail(-2, "M < 0");
    if (want_grad && !out_grad) return fail(-3, "want_grad set but out_grad is NULL");
    if (M == 0) return 0;
    const int L = p->L, n = L + 1;
    if (!theta) {
        // delayedCovariance.jl:3-7: scale > 0 is asserted and rho <= 0 is an error.  The reference wraps the
        // objective in `safewrapper` (:153), i.e. the optimiser sees a penalty instead of the exception; here
        // such rows get info = -1 and loglik = -Inf and are not sent to the device.
    }
    gpcc_ctx* ctx = p->ctx;
    Timer tm;
    reset_stats(ctx);
    const int nd = (int)ctx->ds.size();
    const size_t chunk = 1 << 18;
    int rc = for_each_device(ctx, [&](int di) -> int {
        EvalSlot& s = ctx->ds[di].slot;
        std::vector<int> mine;
        for (int m = di; m < M; m += nd) mine.push_back(m);
        if (p->method == GPCC_METHOD_DENSE && !p->small_path && !want_grad && !theta && L >= 2) {
            // logL-only sweep on the tiled path: bring evaluations with the same hyper-parameters and the same delays of all
            // bands but the last next to each other (structure reuse in large_path.cu); results are scattered back by index
            std::stable_sort(mine.begin(), mine.end(), [&](int x, int y) {
                bool dec;
                bool lt = bits_less(rho[x], rho[y], dec); if (dec) return lt;
                for (int l = 0; l < L; ++l) { lt = bits_less(alpha[(size_t)x * L + l], alpha[(size_t)y * L + l], dec); if (dec) return lt; }
                for (int l = 0; l + 1 < L; ++l) { lt = bits_less(delays[(size_t)x * L + l], delays[(size_t)y * L + l], dec); if (dec) return lt; }
                return false;
            });
        }
        std::vector<double> jac(n);
        for (size_t c0 = 0; c0 < mine.size(); c0 += chunk) {
            const size_t c1 = std::min(mine.size(), c0 + chunk);
            int r = reserve_eval(p, di, c1 - c0);
            if (r) return r;
            std::vector<int> sent;
            sent.reserve(c1 - c0);
            for (size_t c = c0; c < c1; ++c) {
                const int m = mine[c];
                const size_t e = sent.size();
                bool valid = true;
                if (theta) {
                    unpack_theta(theta + (size_t)m * n, L, *o, s.alpha.h + e * L, s.rho.h + e, nullptr);
                } else {
                    std::memcpy(s.alpha.h + e * L, alpha + (size_t)m * L, L * sizeof(double));
                    s.rho.h[e] = rho[m];
                }
                for (int l = 0; l < L; ++l) valid = valid && (s.alpha.h[e * L + l] > 0) && std::isfinite(s.alpha.h[e * L + l]);
                valid = valid && (s.rho.h[e] > 0) && std::isfinite(s.rho.h[e]);
                for (int l = 0; l < L; ++l) valid = valid && std::isfinite(delays[(size_t)m * L + l]);
                if (!valid) {
                    out_ll[m] = -std::numeric_limits<double>::infinity();
                    if (out_info) out_info[m] = -1;
                    if (want_grad) for (int k = 0; k < n; ++k) out_grad[(size_t)m * n + k] = 0.0;
                    continue;
                }
                std::memcpy(s.delays.h + e * L, delays + (size_t)m * L, L * sizeof(double));
                sent.push_back(m);
            }
            if (sent.empty()) continue;
            r = evaluate_on_device(p, di, (int)sent.size(), want_grad);
            if (r) return r;
            for (size_t e = 0; e < sent.size(); ++e) {
                const int m = sent[e];
                out_ll[m] = s.ll.h[e];
                if (out_info) out_info[m] = s.info.h[e];
                if (want_grad) {
                    if (theta) {
                        double a_[LBFGS_MAXN], r_;
                        unpack_theta(theta + (size_t)m * n, L, *o, a_, &r_, jac.data());
                        for (int k = 0; k < n; ++k) out_grad[(size_t)m * n + k] = s.grad.h[e * n + k] * jac[k];
                    } else {
                        std::memcpy(out_grad + (size_t)m * n, s.grad.h + e * n, n * sizeof(double));
                    }
                }
            }
        }
        return 0;
    });
    collect_stats(ctx, p, tm.ms());
    return rc;
}

int gpcc_loglik_batch(gpcc_problem* p, int M, const double* delays, const double* alpha, const double* rho,
                      int want_grad, double* out_ll, double* out_grad, int* out_info) {
    if (!alpha || !rho) return fail(-1, "NULL argument");
    return loglik_batch_impl(p, M, delays, alpha, rho, nullptr, nullptr, want_grad, out_ll, out_grad, out_info);
}

int gpcc_loglik_theta_batch(gpcc_problem* p, int M, const double* delays, const double* theta,
                            const gpcc_fit_options* opt, int want_grad, double* out_ll, double* out_grad,
                            int* out_info) {
    if (!theta) return fail(-1, "NULL argument");
    int rc = check_options(opt);
    if (rc) return rc;
    return loglik_batch_impl(p, M, delays, nullptr, nullptr, theta, opt, want_grad, out_ll, out_grad, out_info);
}

int gpcc_fit_batch(gpcc_problem* p, int M, const double* delays, int P, const double* theta0,
                   const gpcc_fit_options* opt, double* out_ll, double* out_theta, double* out_alpha,
                   double* out_rho, int* out_iters, int* out_nfev, int* out_info) {
    if (!p || !delays || !theta0) return fail(-1, "NULL argument");
    int rc = check_options(opt);
    if (rc) return rc;
    if (M < 0 || P < 1) return fail(-2, "need M >= 0 and P >= 1");
    if (M == 0) return 0;
    for (size_t i = 0; i < (size_t)M * p->L; ++i)
        if (!std::isfinite(delays[i])) return fail(-3, "non-finite delay");
    Timer tm;
    reset_stats(p->ctx);
    FitOutputs out{out_ll, out_theta, out_alpha, out_rho, out_iters, out_nfev, out_info};
    rc = fit_all(p, M, delays, P, theta0, *opt, out);
    collect_stats(p->ctx, p, tm.ms());
    return rc;
}

int gpcc_grid_posterior(gpcc_problem* p, int M, const double* delays, const double* logprior, int P,
                        const double* theta0, const gpcc_fit_options* opt, double* out_ll, double* out_post,
                        double* out_theta, double* out_alpha, double* out_rho, int* out_nfev, int* out_info) {
    if (!p || !delays || !theta0 || !out_post) return fail(-1, "NULL argument");
    int rc = check_options(opt);
    if (rc) return rc;
    if (M < 1 || P < 1) return fail(-2, "need M >= 1 and P >= 1");
    Timer tm;
    reset_stats(p->ctx);
    const int L = p->L, n = L + 1;
    // every output is needed internally: with several ranks the all-gather carries the whole record of a candidate
    std::vector<double> ll_l, th_l, al_l, rh_l;
    std::vector<int> nf_l, in_l;
    GatherIO io;
    io.ll = out_ll ? out_ll : (ll_l.resize(M), ll_l.data());
    io.theta = out_theta ? out_theta : (th_l.resize((size_t)M * n), th_l.data());
    io.alpha = out_alpha ? out_alpha : (al_l.resize((size_t)M * L), al_l.data());
    io.rho = out_rho ? out_rho : (rh_l.resize(M), rh_l.data());
    io.nfev = out_nfev ? out_nfev : (nf_l.resize(M), nf_l.data());
    io.info = out_info ? out_info : (in_l.resize(M), in_l.data());
    FitOutputs out{io.ll, io.theta, io.alpha, io.rho, nullptr, io.nfev, io.info};
    rc = fit_all(p, M, delays, P, theta0, *opt, out);
    if (rc) return rc;
    // all-gather of the per-device slices (NCCL when the grid spans several devices or ranks) + log-sum-exp on device
    rc = posterior_on_devices(p->ctx, L, M, io, logprior, out_post);
    if (rc) return rc;
    if (p->ctx->world > 1)        // alpha, rho of the other ranks' candidates follow from their gathered theta (unpack, :235)
        for (int m = 0; m < M; ++m) {
            if (io.info[m] == LbfgsState::NO_START) {
                for (int l = 0; l < L; ++l) io.alpha[(size_t)m * L + l] = std::numeric_limits<double>::quiet_NaN();
                io.rho[m] = std::numeric_limits<double>::quiet_NaN();
            } else unpack_theta(io.theta + (size_t)m * n, L, *opt, io.alpha + (size_t)m * L, io.rho + m, nullptr);
        }
    collect_stats(p->ctx, p, tm.ms());
    return rc;
}

int gpcc_comm_unique_id(char* out_id128) {
    if (!out_id128) return fail(-1, "NULL argument");
    std::string err;
    if (nccl_bridge_unique_id(out_id128, err)) return fail(2000, "NCCL unavailable: " + err);
    return 0;
}

int gpcc_ctx_comm_init_rank(gpcc_ctx* ctx, int world, int rank, const char* id128) {
    if (!ctx || !id128) return fail(-1, "NULL argument");
    if (world < 1 || rank < 0 || rank >= world) return fail(-2, "need 0 <= rank < world");
    if (ctx->ds.size() != 1) return fail(-3, "a context that joins a multi-process communicator must own exactly one device");
    if (ctx->nccl) { nccl_bridge_destroy(ctx->nccl); ctx->nccl = nullptr; }
    ctx->world = 1; ctx->rank = 0;
    if (world == 1) return 0;
    std::string err;
    ctx->nccl = nccl_bridge_create_rank(ctx->ds[0].dev, world, rank, id128, err);
    if (!ctx->nccl) return fail(2000, "NCCL unavailable for the multi-process allgather: " + err);
    ctx->world = world; ctx->rank = rank;
    return 0;
}

int gpcc_getprobabilities(gpcc_ctx* ctx, int M, const double* loglik, const double* logprior, double* out_post) {
    if (!ctx || !loglik || !out_post) return fail(-1, "NULL argument");
    if (M < 1) return fail(-2, "M < 1");
    DeviceState& s = ctx->ds[0];
    CUDA_TRY(cudaSetDevice(s.dev));
    cudaStream_t st = s.stream.get();
    // persistent buffers: cudaMalloc/cudaFree serialise against every other context on the box (and stall for hundreds
    // of milliseconds when several ranks with NCCL peer mappings hit them at once), so the hot path never calls them
    CUDA_TRY(s.post_ll.reserve(M));
    CUDA_TRY(s.post_out.reserve(M));
    if (logprior) CUDA_TRY(s.post_prior.reserve(M));
    std::memcpy(s.post_ll.h, loglik, (size_t)M * sizeof(double));
    CUDA_TRY(cudaMemcpyAsync(s.post_ll.d, s.post_ll.h, (size_t)M * sizeof(double), cudaMemcpyHostToDevice, st));
    if (logprior) {
        std::memcpy(s.post_prior.h, logprior, (size_t)M * sizeof(double));
        CUDA_TRY(cudaMemcpyAsync(s.post_prior.d, s.post_prior.h, (size_t)M * sizeof(double), cudaMemcpyHostToDevice, st));
    }
    CUDA_TRY(posterior_launch(M, s.post_ll.d, logprior ? s.post_prior.d : nullptr, s.post_out.d, st));
    CUDA_TRY(cudaMemcpyAsync(s.post_out.h, s.post_out.d, (size_t)M * sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    std::memcpy(out_post, s.post_out.h, (size_t)M * sizeof(double));
    return 0;
}

}  // extern "C"

// ---- posterior over the grid: allgather + log-sum-exp ---------------------------------------------------
namespace gpcc {

int posterior_on_devices(gpcc_ctx* ctx, int L, int M, const GatherIO& io, const double* logprior, double* out_post) {
    const int nd = (int)ctx->ds.size();
    const int G = ctx->world * nd;
    if (G == 1) return gpcc_getprobabilities(ctx, M, io.ll, logprior, out_post);
    // Global device g owns the strided slice m = g, g+G, ...  Every device packs its slice into records
    //   [loglik, joint = loglik + logprior, theta (L+1), nfev, info]
    // padded to a common length, reduces the joint column to (max, sum exp) on the device, and ONE ncclAllGather over
    // NVLink distributes records and partials; the combine after it is G elements (src/getprobabilities.jl:14-16).
    const int n = L + 1, REC = n + 4, JCOL = 1;
    const int per = (M + G - 1) / G;
    const size_t blk = (size_t)per * REC + 2;
    if (!ctx->nccl) {
        std::vector<int> devs;
        for (auto& s : ctx->ds) devs.push_back(s.dev);
        std::string err;
        ctx->nccl = nccl_bridge_create(devs, err);
        // one process holds every device's results on the host already: without NCCL the posterior is still computed on
        // device 0 (a multi-process communicator cannot do without it and fails in gpcc_ctx_comm_init_rank instead)
        if (!ctx->nccl) return gpcc_getprobabilities(ctx, M, io.ll, logprior, out_post);
    }
    std::vector<double*> d_send(nd), d_recv(nd);
    std::vector<cudaStream_t> streams(nd);
    const double ninf = -std::numeric_limits<double>::infinity();
    for (int di = 0; di < nd; ++di) {
        DeviceState& s = ctx->ds[di];
        CUDA_TRY(cudaSetDevice(s.dev));
        CUDA_TRY(s.gat_send.reserve(blk));
        CUDA_TRY(s.gat_recv.reserve(blk * G));
        const int g = ctx->rank * nd + di;
        double* h = s.gat_send.h;
        for (int k = 0; k < per; ++k) {
            const int m = g + k * G;
            double* r = h + (size_t)k * REC;
            if (m < M) {
                r[0] = io.ll[m];
                r[1] = io.ll[m] + (logprior ? logprior[m] : 1.0);            // joint (getprobabilities.jl:3,14)
                std::memcpy(r + 2, io.theta + (size_t)m * n, n * sizeof(double));
                r[2 + n] = (double)io.nfev[m];
                r[3 + n] = (double)io.info[m];
            } else {
                r[0] = ninf; r[1] = ninf;
                for (int q = 2; q < REC; ++q) r[q] = 0.0;
            }
        }
        CUDA_TRY(cudaMemcpyAsync(s.gat_send.d, h, (size_t)per * REC * sizeof(double), cudaMemcpyHostToDevice, s.stream.get()));
        CUDA_TRY(posterior_partial_launch(per, REC, JCOL, s.gat_send.d, s.stream.get()));
        d_send[di] = s.gat_send.d; d_recv[di] = s.gat_recv.d; streams[di] = s.stream.get();
    }
    std::string err;
    if (nccl_bridge_allgather(ctx->nccl, d_send, d_recv, (int)blk, streams, err)) return fail(2001, "ncclAllGather: " + err);
    DeviceState& s0 = ctx->ds[0];
    CUDA_TRY(cudaSetDevice(s0.dev));
    cudaStream_t st0 = s0.stream.get();
    CUDA_TRY(s0.gat_post.reserve((size_t)per * G));
    CUDA_TRY(posterior_combine_launch(G, per, REC, JCOL, s0.gat_recv.d, s0.gat_post.d, st0));
    CUDA_TRY(cudaMemcpyAsync(s0.gat_post.h, s0.gat_post.d, (size_t)per * G * sizeof(double), cudaMemcpyDeviceToHost, st0));
    CUDA_TRY(cudaMemcpyAsync(s0.gat_recv.h, s0.gat_recv.d, blk * G * sizeof(double), cudaMemcpyDeviceToHost, st0));
    CUDA_TRY(cudaStreamSynchronize(st0));
    for (int g = 0; g < G; ++g)
        for (int k = 0; k < per; ++k) {
            const int m = g + k * G;
            if (m >= M) continue;
            out_post[m] = s0.gat_post.h[(size_t)g * per + k];
            if (ctx->world > 1) {      // the other ranks' candidates arrive through the gather
                const double* r = s0.gat_recv.h + g * blk + (size_t)k * REC;
                io.ll[m] = r[0];
                std::memcpy(io.theta + (size_t)m * n, r + 2, n * sizeof(double));
                io.nfev[m] = (int)r[2 + n];
                io.info[m] = (int)r[3 + n];
            }
        }
    for (auto& s : ctx->ds) s.launches += 2;
    return 0;
}

}  // namespace gpcc

namespace gpcc {

int statespace_postb(gpcc_problem* p, const double* delays, const double* alpha, double rho, double* out_mu, double* out_Sigma) {
    const int L = p->L;
    DeviceState& s = p->ctx->ds[0];
    gpcc_problem::PerDev& d = p->pd[0];
    CUDA_TRY(cudaSetDevice(s.dev));
    int rc = reserve_eval(p, 0, 1);
    if (rc) return rc;
    EvalSlot& q = s.slot;
    cudaStream_t st = s.stream.get();
    CUDA_TRY(cudaStreamSynchronize(st));          // the pinned staging may still be read by an earlier call
    std::memcpy(q.delays.h, delays, L * sizeof(double));
    std::memcpy(q.alpha.h, alpha, L * sizeof(double));
    q.rho.h[0] = rho;
    CUDA_TRY(cudaMemcpyAsync(q.delays.d, q.delays.h, L * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(q.alpha.d, q.alpha.h, L * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(q.rho.d, q.rho.h, sizeof(double), cudaMemcpyHostToDevice, st));
    EvalBatch b;
    b.M = 1; b.delays = q.delays.d; b.alpha = q.alpha.d; b.rho = q.rho.d; b.want_grad = 0;
    b.ll = q.ll.d; b.grad = q.grad.d; b.info = q.info.d;
    CUDA_TRY(statespace_launch(p->kernel_id, d.ssp, b, d.ss_postb.d, st));
    const size_t n = (size_t)L + (size_t)L * L;
    CUDA_TRY(cudaMemcpyAsync(d.ss_postb.h, d.ss_postb.d, n * sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(q.info.h, q.info.d, sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    s.launches += 1;
    if (q.info.h[0] != 0) return fail(-6, "the filter met a non-positive innovation variance for these hyper-parameters");
    std::memcpy(out_mu, d.ss_postb.h, L * sizeof(double));
    std::memcpy(out_Sigma, d.ss_postb.h + L, (size_t)L * L * sizeof(double));    // symmetric: the layout does not matter
    return 0;
}

}  // namespace gpcc

// ---- fit state of the state-space method (gpcc_ss_state_*): O(N) memory, predictions in O(D^3) per test point ----
struct gpcc_ss_state {
    int dev = 0, kernel_id = 0, N = 0, L = 0, D = 0;
    SSProblem prior;                    // N, L, band_start, mu_b, Sigma_b of the training problem (no data pointers)
    std::vector<double> tr_t, tr_r, tr_s2;   // training data, each band sorted by t: merged with the test points of a call
    std::vector<int> tr_ord;            // input index of every sorted training point (the deviates of gpcc_ss_state_sample)
    std::vector<double> h_hyp;          // host copy of hyp
    double ll_train = 0.0;
    Stream stream;
    DevArray<double> hyp;               // delays [L], alpha [L], rho
    DevArray<double> st_t, st_m, st_P, st_lam, st_Lam;
    DevArray<int> st_band;
    SSStore st;
    // scratch of the calls, kept between calls
    DevArray<double> tt, mu, sd, mt, mr, ms2, ll;
    DevArray<int> bt, info;
    // gpcc_ss_state_sample: the per-step records, built by its first call and kept (N (d^2 + D + 3) doubles + N ints), and
    // the scratch of its calls (the prior sampler over the merged problem, one chunk of the mean passes)
    DevArray<double> ps_rec;
    DevArray<int> ps_in;
    DevArray<double> ps_f, ps_z, ps_bs, ps_dv, ps_mbuf, ps_lbuf, ps_tw, ps_out, ps_step, ps_aggA, ps_aggc;
    DevArray<int> ps_perm, ps_ints, ps_need, ps_mpos, ps_lpos, ps_tstep;
    ~gpcc_ss_state() { cudaSetDevice(dev); }
};

namespace {

int ss_state_create(gpcc_problem* p, const double* delays, const double* alpha, double rho, gpcc_ss_state** out) {
    const int N = p->N, L = p->L, d = p->kernel_id == GPCC_KERNEL_OU ? 1 : p->kernel_id == GPCC_KERNEL_MATERN32 ? 2 : 3;
    const size_t D = (size_t)(d + L), NP = D * (D + 1) / 2;
    const gpcc_problem::PerDev& pd = p->pd[0];
    CUDA_TRY(cudaSetDevice(pd.dev));
    std::unique_ptr<gpcc_ss_state> s(new gpcc_ss_state());
    s->dev = pd.dev; s->kernel_id = p->kernel_id; s->N = N; s->L = L; s->D = (int)D;
    s->prior = pd.ssp;
    s->prior.t = s->prior.r = s->prior.s2 = nullptr;
    sort_bands(p, s->tr_t, s->tr_r, s->tr_s2, &s->tr_ord);
    CUDA_TRY(create_stream(s->stream, 0));
    cudaStream_t st = s->stream.get();
    std::vector<double> h(2 * L + 1);
    std::memcpy(h.data(), delays, L * sizeof(double));
    std::memcpy(h.data() + L, alpha, L * sizeof(double));
    h[2 * L] = rho;
    s->h_hyp = h;
    CUDA_TRY(s->hyp.reserve(h.size()));
    CUDA_TRY(s->st_t.reserve(N));
    CUDA_TRY(s->st_band.reserve(N));
    CUDA_TRY(s->st_m.reserve((size_t)N * D));
    CUDA_TRY(s->st_P.reserve((size_t)N * NP));
    CUDA_TRY(s->st_lam.reserve((size_t)N * D));
    CUDA_TRY(s->st_Lam.reserve((size_t)N * NP));
    CUDA_TRY(s->ll.reserve(1));
    CUDA_TRY(s->info.reserve(1));
    s->st = SSStore{s->st_t.d, s->st_band.d, s->st_m.d, s->st_P.d, s->st_lam.d, s->st_Lam.d};
    CUDA_TRY(cudaMemcpyAsync(s->hyp.d, h.data(), h.size() * sizeof(double), cudaMemcpyHostToDevice, st));
    // the problem's sorted device copies are read only here: the state keeps what its calls need
    CUDA_TRY(statespace_store_launch(s->kernel_id, pd.ssp, s->hyp.d, s->ll.d, s->info.d, s->st, st));
    int info = 0;
    CUDA_TRY(cudaMemcpyAsync(&s->ll_train, s->ll.d, sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(&info, s->info.d, sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (info != 0) return fail(-6, "the filter met a non-positive innovation variance for these hyper-parameters");
    *out = s.release();
    return 0;
}

// The argument checks of the calls that take a state-space problem and its hyper-parameters.
int ss_check_hyper(const gpcc_problem* p, const double* delays, const double* alpha, double rho) {
    if (!p || !delays || !alpha) return fail(-1, "NULL argument");
    if (p->method != GPCC_METHOD_STATESPACE) return fail(-5, "the problem is not in GPCC_METHOD_STATESPACE (gpcc_problem_set_method)");
    for (int l = 0; l < p->L; ++l) {
        if (!(alpha[l] > 0) || !std::isfinite(alpha[l])) return fail(-2, "all(scale .> 0) violated (delayedCovariance.jl:3)");
        if (!std::isfinite(delays[l])) return fail(-3, "non-finite delay");
    }
    if (!(rho > 0) || !std::isfinite(rho)) return fail(-4, "rho is <= 0 (delayedCovariance.jl:5-7)");
    return 0;
}

// gpcc_ss_sample after its checks: the five kernels of ss_sample.cu on the first device and stream.
int ss_sample(gpcc_problem* p, const double* delays, const double* alpha, double rho, unsigned long long seed, int nsamples,
              const double* z_in, double* out_f, double* out_z) {
    const int N = p->N, L = p->L, d = p->kernel_id == GPCC_KERNEL_OU ? 1 : p->kernel_id == GPCC_KERNEL_MATERN32 ? 2 : 3;
    const size_t nf = (size_t)nsamples * N, nz = nf * (d + 1);
    gpcc_problem::PerDev& pd = p->pd[0];
    DeviceState& ds = p->ctx->ds[0];
    CUDA_TRY(cudaSetDevice(pd.dev));
    cudaStream_t st = ds.stream.get();
    SSSampleBuffers& b = pd.ss_smp;
    size_t n_step, n_aggA, n_aggc;
    statespace_sample_scratch(p->kernel_id, N, nsamples, n_step, n_aggA, n_aggc);
    CUDA_TRY(b.ints.reserve(2 * (size_t)N));
    CUDA_TRY(b.step.reserve(n_step));
    CUDA_TRY(b.aggA.reserve(n_aggA));
    CUDA_TRY(b.aggc.reserve(n_aggc));
    CUDA_TRY(b.f.reserve(nf));
    if (z_in || out_z) CUDA_TRY(b.z.reserve(nz));
    if (z_in) CUDA_TRY(cudaMemcpyAsync(b.z.d, z_in, nz * sizeof(double), cudaMemcpyHostToDevice, st));
    SSSampleArgs a;
    for (int l = 0; l < L; ++l) { a.tau[l] = delays[l]; a.alpha[l] = alpha[l]; }
    a.rho = rho; a.seed = seed; a.nsamples = nsamples; a.perm = pd.ss_perm.d;
    a.zin = z_in ? b.z.d : nullptr;
    a.zout = out_z && !z_in ? b.z.d : nullptr;
    a.f = b.f.d;
    SSSampleScratch sc{b.ints.d, b.ints.d + N, b.step.d, b.aggA.d, b.aggc.d};
    CUDA_TRY(statespace_sample_launch(p->kernel_id, pd.ssp, a, sc, st));
    CUDA_TRY(cudaMemcpyAsync(out_f, b.f.d, nf * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (out_z) CUDA_TRY(cudaMemcpyAsync(out_z, b.z.d, nz * sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    ds.launches += 5;
    return 0;
}

// Test points of one call: counts, band of every point in input order, and the checks shared by both calls.
int ss_test_points(const gpcc_ss_state* s, const int* ntest_per_band, const double* ttest, std::vector<int>& bt) {
    if (!s || !ntest_per_band) return fail(-1, "NULL argument");
    long long NT = 0;
    for (int l = 0; l < s->L; ++l) {
        if (ntest_per_band[l] < 0) return fail(-5, "negative test count");
        NT += ntest_per_band[l];
    }
    if (NT > (1LL << 30)) return fail(-7, "too many test points for one call");
    if (NT > 0 && !ttest) return fail(-1, "NULL argument");
    bt.resize((size_t)NT);
    for (int l = 0, k = 0; l < s->L; ++l)
        for (int i = 0; i < ntest_per_band[l]; ++i, ++k) {
            if (!std::isfinite(ttest[k])) return fail(-3, "non-finite test time");
            bt[k] = l;
        }
    return 0;
}

// Records of gpcc_ss_state_sample (first call): the sorted training data go to the device for the rank and record kernels
// only; the state keeps the records.
int ss_post_records(gpcc_ss_state* s) {
    const size_t N = (size_t)s->N;
    cudaStream_t st = s->stream.get();
    DevArray<double> t, r, s2;
    DevArray<int> perm, order;
    CUDA_TRY(t.reserve(N));
    CUDA_TRY(r.reserve(N));
    CUDA_TRY(s2.reserve(N));
    CUDA_TRY(perm.reserve(N));
    CUDA_TRY(order.reserve(N));
    CUDA_TRY(s->ps_rec.reserve(N * statespace_post_record_width(s->kernel_id, s->L)));
    CUDA_TRY(s->ps_in.reserve(N));
    CUDA_TRY(cudaMemcpyAsync(t.d, s->tr_t.data(), N * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(r.d, s->tr_r.data(), N * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(s2.d, s->tr_s2.data(), N * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(perm.d, s->tr_ord.data(), N * sizeof(int), cudaMemcpyHostToDevice, st));
    SSProblem q = s->prior;
    q.t = t.d; q.r = r.d; q.s2 = s2.d;
    CUDA_TRY(statespace_post_records_launch(s->kernel_id, q, s->hyp.d, s->h_hyp.data(), s->st, perm.d, order.d, s->ps_rec.d,
                                            s->ps_in.d, st));
    CUDA_TRY(cudaStreamSynchronize(st));      // before the temporaries are freed
    return 0;
}

constexpr size_t PS_CHUNK_BYTES = size_t(1) << 30;   // scratch of one chunk of samples of gpcc_ss_state_sample
constexpr unsigned PS_STREAM_TAG = 0x53535053u;      // "SSPS": apart from gpcc_ss_sample's "SSMP" and the dense "GPCC"

// gpcc_ss_state_sample after its checks.  The merged problem of the prior draw: per band the sorted training points and the
// sorted test points, training first on ties (as gpcc_ss_state_predict_loglik merges them), test points with sigma^2 = 1e-8;
// its input indices are the training input order, then N + the test input order.
int ss_state_sample(gpcc_ss_state* s, const int* ntest_per_band, const double* ttest, const std::vector<int>& bt,
                    unsigned long long seed, int nsamples, const double* z_in, double* out_f, double* out_z) {
    const int L = s->L, N = s->N, NT = (int)bt.size(), NM = N + NT;
    const int d = s->kernel_id == GPCC_KERNEL_OU ? 1 : s->kernel_id == GPCC_KERNEL_MATERN32 ? 2 : 3, D = d + L;
    const size_t zp = (size_t)NM * (d + 1);             // point deviates per sample
    std::vector<double> mt(NM), ms2(NM);
    std::vector<int> mperm(NM);
    SSProblem q = s->prior;
    q.N = NM;
    std::vector<size_t> ord;
    size_t k = 0, first = 0;
    for (int l = 0; l < L; ++l) {
        const size_t nt = (size_t)ntest_per_band[l];
        ord.resize(nt);
        for (size_t i = 0; i < nt; ++i) ord[i] = first + i;
        std::stable_sort(ord.begin(), ord.end(), [&](size_t a, size_t b) { return ttest[a] < ttest[b]; });
        q.band_start[l] = (int)k;
        size_t a = s->prior.band_start[l], b = 0;
        const size_t ae = s->prior.band_start[l + 1];
        while (a < ae || b < nt) {
            if (b == nt || (a < ae && s->tr_t[a] <= ttest[ord[b]])) {
                mt[k] = s->tr_t[a]; ms2[k] = s->tr_s2[a]; mperm[k] = s->tr_ord[a]; ++a;
            } else {
                const size_t j = ord[b++];
                mt[k] = ttest[j]; ms2[k] = 1e-8; mperm[k] = N + (int)j;
            }
            ++k;
        }
        first += nt;
    }
    q.band_start[L] = (int)k;

    CUDA_TRY(cudaSetDevice(s->dev));
    cudaStream_t st = s->stream.get();
    if (!s->ps_rec.d) {
        int rc = ss_post_records(s);
        if (rc) return rc;
    }
    // samples per chunk: the per-sample scratch of the prior draw and of the mean passes within PS_CHUNK_BYTES
    const size_t tiles = ((size_t)NM + 63) / 64;
    const size_t per = (size_t)NM + (z_in || out_z ? zp + L : 0) + L + (size_t)N + 2 * (size_t)NT * D + NT + tiles * d;
    const int C = (int)std::max<size_t>(1, std::min<size_t>((size_t)nsamples, PS_CHUNK_BYTES / (per * sizeof(double))));
    size_t n_step, n_aggA, n_aggc;
    statespace_sample_scratch(s->kernel_id, NM, C, n_step, n_aggA, n_aggc);
    CUDA_TRY(s->mt.reserve(NM));
    CUDA_TRY(s->ms2.reserve(NM));
    CUDA_TRY(s->ps_perm.reserve(NM));
    CUDA_TRY(s->ps_ints.reserve(2 * (size_t)NM));
    CUDA_TRY(s->ps_step.reserve(n_step));
    CUDA_TRY(s->ps_aggA.reserve(n_aggA));
    CUDA_TRY(s->ps_aggc.reserve(n_aggc));
    CUDA_TRY(s->ps_f.reserve((size_t)C * NM));
    if (z_in || out_z) CUDA_TRY(s->ps_z.reserve((size_t)C * (zp + L)));
    CUDA_TRY(s->ps_bs.reserve((size_t)C * L));
    CUDA_TRY(s->ps_dv.reserve((size_t)C * N));
    CUDA_TRY(s->ps_mbuf.reserve((size_t)C * NT * D));
    CUDA_TRY(s->ps_lbuf.reserve((size_t)C * NT * D));
    CUDA_TRY(s->ps_out.reserve((size_t)C * NT));
    CUDA_TRY(s->ps_tw.reserve((size_t)NT * 2 * D));
    CUDA_TRY(s->ps_tstep.reserve(NT));
    CUDA_TRY(s->ps_need.reserve(N));
    CUDA_TRY(s->ps_mpos.reserve(N));
    CUDA_TRY(s->ps_lpos.reserve(N));
    CUDA_TRY(s->tt.reserve(NT));
    CUDA_TRY(s->bt.reserve(NT));
    CUDA_TRY(cudaMemcpyAsync(s->mt.d, mt.data(), NM * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(s->ms2.d, ms2.data(), NM * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(s->ps_perm.d, mperm.data(), NM * sizeof(int), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(s->tt.d, ttest, NT * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(s->bt.d, bt.data(), NT * sizeof(int), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemsetAsync(s->ps_need.d, 0, N * sizeof(int), st));
    q.t = s->mt.d; q.s2 = s->ms2.d; q.r = nullptr;
    CUDA_TRY(statespace_post_locate_launch(s->kernel_id, s->prior, s->hyp.d, s->st, NT, s->tt.d, s->bt.d, s->ps_tstep.d,
                                           s->ps_tw.d, s->ps_need.d, st));
    SSSampleArgs sa;
    for (int l = 0; l < L; ++l) { sa.tau[l] = s->h_hyp[l]; sa.alpha[l] = s->h_hyp[L + l]; }
    sa.rho = s->h_hyp[2 * L]; sa.seed = seed; sa.tag = PS_STREAM_TAG; sa.perm = s->ps_perm.d; sa.f = s->ps_f.d;
    SSSampleScratch sc{s->ps_ints.d, s->ps_ints.d + NM, s->ps_step.d, s->ps_aggA.d, s->ps_aggc.d};
    SSPostArgs pa;
    pa.N = N; pa.NT = NT; pa.NM = NM; pa.L = L; pa.seed = seed; pa.tag = PS_STREAM_TAG;
    for (int l = 0; l < L; ++l) { pa.mub[l] = s->prior.mub[l]; pa.sqrt_sigmab[l] = std::sqrt(s->prior.Sigmab[l]); }
    pa.rec = s->ps_rec.d; pa.in = s->ps_in.d; pa.band = s->st.band;
    pa.tstep = s->ps_tstep.d; pa.tw = s->ps_tw.d; pa.bt = s->bt.d; pa.need = s->ps_need.d;
    pa.mpos = s->ps_mpos.d; pa.lpos = s->ps_lpos.d; pa.f = s->ps_f.d; pa.bs = s->ps_bs.d; pa.dv = s->ps_dv.d;
    pa.mbuf = s->ps_mbuf.d; pa.lbuf = s->ps_lbuf.d; pa.out = s->ps_out.d;
    for (int s0 = 0; s0 < nsamples; s0 += C) {
        const int c = std::min(C, nsamples - s0);
        double* zb = (z_in || out_z) ? s->ps_z.d + (size_t)c * zp : nullptr;    // [c][L] after the [c][NM][d+1] points
        if (z_in) {
            CUDA_TRY(cudaMemcpyAsync(s->ps_z.d, z_in + (size_t)s0 * zp, (size_t)c * zp * sizeof(double), cudaMemcpyHostToDevice, st));
            CUDA_TRY(cudaMemcpyAsync(zb, z_in + (size_t)nsamples * zp + (size_t)s0 * L, (size_t)c * L * sizeof(double),
                                     cudaMemcpyHostToDevice, st));
        }
        sa.nsamples = c; sa.sample0 = s0;
        sa.zin = z_in ? s->ps_z.d : nullptr;
        sa.zout = out_z && !z_in ? s->ps_z.d : nullptr;
        CUDA_TRY(statespace_sample_launch(s->kernel_id, q, sa, sc, st));
        pa.C = c; pa.sample0 = s0;
        pa.zin_b = z_in ? zb : nullptr;
        pa.zout_b = out_z && !z_in ? zb : nullptr;
        CUDA_TRY(statespace_post_chunk_launch(s->kernel_id, pa, st));
        CUDA_TRY(cudaMemcpyAsync(out_f + (size_t)s0 * NT, s->ps_out.d, (size_t)c * NT * sizeof(double), cudaMemcpyDeviceToHost, st));
        if (out_z) {
            CUDA_TRY(cudaMemcpyAsync(out_z + (size_t)s0 * zp, s->ps_z.d, (size_t)c * zp * sizeof(double), cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaMemcpyAsync(out_z + (size_t)nsamples * zp + (size_t)s0 * L, zb, (size_t)c * L * sizeof(double),
                                     cudaMemcpyDeviceToHost, st));
        }
    }
    CUDA_TRY(cudaStreamSynchronize(st));
    return 0;
}

}  // namespace

extern "C" {

int gpcc_ss_state_create(gpcc_problem* p, const double* delays, const double* alpha, double rho, gpcc_ss_state** out) {
    if (!out) return fail(-1, "out is NULL");
    *out = nullptr;
    int rc = ss_check_hyper(p, delays, alpha, rho);
    if (rc) return rc;
    return ss_state_create(p, delays, alpha, rho, out);
}

int gpcc_ss_state_destroy(gpcc_ss_state* s) {
    delete s;
    return 0;
}

int gpcc_ss_state_predict(gpcc_ss_state* s, const int* ntest_per_band, const double* ttest, double* out_mu, double* out_sd) {
    std::vector<int> bt;
    int rc = ss_test_points(s, ntest_per_band, ttest, bt);
    if (rc) return rc;
    const size_t NT = bt.size();
    if (NT == 0) return 0;
    if (!out_mu) return fail(-1, "NULL argument");
    CUDA_TRY(cudaSetDevice(s->dev));
    cudaStream_t st = s->stream.get();
    CUDA_TRY(s->tt.reserve(NT));
    CUDA_TRY(s->bt.reserve(NT));
    CUDA_TRY(s->mu.reserve(NT));
    if (out_sd) CUDA_TRY(s->sd.reserve(NT));
    CUDA_TRY(cudaMemcpyAsync(s->tt.d, ttest, NT * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(s->bt.d, bt.data(), NT * sizeof(int), cudaMemcpyHostToDevice, st));
    CUDA_TRY(statespace_predict_launch(s->kernel_id, s->prior, s->hyp.d, s->st, (int)NT, s->tt.d, s->bt.d, s->mu.d,
                                       out_sd ? s->sd.d : nullptr, st));
    CUDA_TRY(cudaMemcpyAsync(out_mu, s->mu.d, NT * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (out_sd) CUDA_TRY(cudaMemcpyAsync(out_sd, s->sd.d, NT * sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return 0;
}

// log p(ytest | training data) = ll(train + test) - ll(train): one filter over the training points merged with the test points
// (per band, both sorted by t, training first on ties), each test point with noise sigmatest^2 + 1e-8 (the jitter of the
// predictive covariance).  info > 0: 1-based merged position of the first non-positive innovation variance, ll = -Inf.
int gpcc_ss_state_predict_loglik(gpcc_ss_state* s, const int* ntest_per_band, const double* ttest, const double* ytest,
                                 const double* sigmatest, double* out_ll, int* out_info) {
    std::vector<int> bt;
    int rc = ss_test_points(s, ntest_per_band, ttest, bt);
    if (rc) return rc;
    if (!out_ll) return fail(-1, "NULL argument");
    const size_t NT = bt.size();
    if (NT == 0) { *out_ll = 0.0; if (out_info) *out_info = 0; return 0; }
    if (!ytest || !sigmatest) return fail(-1, "NULL argument");
    for (size_t k = 0; k < NT; ++k) {
        if (!std::isfinite(ytest[k]) || !std::isfinite(sigmatest[k])) return fail(-3, "non-finite test value");
        if (sigmatest[k] < 0) return fail(-4, "sigmatest < 0");
    }
    const int L = s->L;
    const size_t NM = (size_t)s->N + NT;
    if (NM > (size_t)std::numeric_limits<int>::max()) return fail(-7, "too many test points for one call");
    std::vector<double> mt(NM), mr(NM), ms2(NM);
    SSProblem q = s->prior;
    q.N = (int)NM;
    std::vector<size_t> ord;
    size_t k = 0, first = 0;
    for (int l = 0; l < L; ++l) {
        const size_t nt = (size_t)ntest_per_band[l];
        ord.resize(nt);
        for (size_t i = 0; i < nt; ++i) ord[i] = first + i;
        std::stable_sort(ord.begin(), ord.end(), [&](size_t a, size_t b) { return ttest[a] < ttest[b]; });
        q.band_start[l] = (int)k;
        size_t a = s->prior.band_start[l], b = 0;
        const size_t ae = s->prior.band_start[l + 1];
        while (a < ae || b < nt) {
            if (b == nt || (a < ae && s->tr_t[a] <= ttest[ord[b]])) {
                mt[k] = s->tr_t[a]; mr[k] = s->tr_r[a]; ms2[k] = s->tr_s2[a]; ++a;
            } else {
                const size_t j = ord[b++];
                mt[k] = ttest[j]; mr[k] = ytest[j] - s->prior.mub[l]; ms2[k] = sigmatest[j] * sigmatest[j] + 1e-8;
            }
            ++k;
        }
        first += nt;
    }
    q.band_start[L] = (int)k;
    CUDA_TRY(cudaSetDevice(s->dev));
    cudaStream_t st = s->stream.get();
    CUDA_TRY(s->mt.reserve(NM));
    CUDA_TRY(s->mr.reserve(NM));
    CUDA_TRY(s->ms2.reserve(NM));
    CUDA_TRY(cudaMemcpyAsync(s->mt.d, mt.data(), NM * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(s->mr.d, mr.data(), NM * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(s->ms2.d, ms2.data(), NM * sizeof(double), cudaMemcpyHostToDevice, st));
    q.t = s->mt.d; q.r = s->mr.d; q.s2 = s->ms2.d;
    EvalBatch b;
    b.M = 1; b.delays = s->hyp.d; b.alpha = s->hyp.d + L; b.rho = s->hyp.d + 2 * L; b.want_grad = 0;
    b.ll = s->ll.d; b.info = s->info.d;
    CUDA_TRY(statespace_launch(s->kernel_id, q, b, nullptr, st));
    double ll = 0.0;
    int info = 0;
    CUDA_TRY(cudaMemcpyAsync(&ll, s->ll.d, sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(&info, s->info.d, sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    *out_ll = info ? -std::numeric_limits<double>::infinity() : ll - s->ll_train;
    if (out_info) *out_info = info;
    return 0;
}

int gpcc_ss_state_sample(gpcc_ss_state* s, const int* ntest_per_band, const double* ttest, unsigned long long seed, int nsamples,
                         const double* z_in, double* out_f, double* out_z) {
    std::vector<int> bt;
    int rc = ss_test_points(s, ntest_per_band, ttest, bt);
    if (rc) return rc;
    if (nsamples < 1) return fail(-7, "nsamples < 1");
    const size_t NT = bt.size();
    if (NT == 0) return 0;
    if (!out_f) return fail(-1, "NULL argument");
    const size_t NM = (size_t)s->N + NT;
    if (NM > (size_t)std::numeric_limits<int>::max()) return fail(-7, "too many test points for one call");
    if (z_in) {
        const size_t d = s->kernel_id == GPCC_KERNEL_OU ? 1 : s->kernel_id == GPCC_KERNEL_MATERN32 ? 2 : 3;
        const size_t nz = (size_t)nsamples * (NM * (d + 1) + s->L);
        for (size_t k = 0; k < nz; ++k)
            if (!std::isfinite(z_in[k])) return fail(-8, "non-finite deviate in z_in");
    }
    return ss_state_sample(s, ntest_per_band, ttest, bt, seed, nsamples, z_in, out_f, out_z);
}

int gpcc_ss_sample(gpcc_problem* p, const double* delays, const double* alpha, double rho, unsigned long long seed, int nsamples,
                   const double* z_in, double* out_f, double* out_z) {
    if (!out_f) return fail(-1, "NULL argument");
    int rc = ss_check_hyper(p, delays, alpha, rho);
    if (rc) return rc;
    if (nsamples < 1) return fail(-7, "nsamples < 1");
    if (z_in) {
        const size_t d = p->kernel_id == GPCC_KERNEL_OU ? 1 : p->kernel_id == GPCC_KERNEL_MATERN32 ? 2 : 3;
        const size_t nz = (size_t)nsamples * p->N * (d + 1);
        for (size_t k = 0; k < nz; ++k)
            if (!std::isfinite(z_in[k])) return fail(-8, "non-finite deviate in z_in");
    }
    return ss_sample(p, delays, alpha, rho, seed, nsamples, z_in, out_f, out_z);
}

}  // extern "C"
