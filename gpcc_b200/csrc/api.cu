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
    cudaStream_t stream = s.stream;
    CUDA_TRY(cudaMemcpyAsync(q.delays.d, q.delays.h, (size_t)M * L * sizeof(double), cudaMemcpyHostToDevice, stream));
    CUDA_TRY(cudaMemcpyAsync(q.alpha.d, q.alpha.h, (size_t)M * L * sizeof(double), cudaMemcpyHostToDevice, stream));
    CUDA_TRY(cudaMemcpyAsync(q.rho.d, q.rho.h, (size_t)M * sizeof(double), cudaMemcpyHostToDevice, stream));
    EvalBatch b;
    b.M = M; b.delays = q.delays.d; b.alpha = q.alpha.d; b.rho = q.rho.d; b.want_grad = want_grad;
    b.ll = q.ll.d; b.grad = q.grad.d; b.info = q.info.d;
    b.h_delays = q.delays.h; b.h_alpha = q.alpha.h; b.h_rho = q.rho.h;
    const bool prof = p->ctx->profiling;
    if (p->small_path) {
        if (prof) CUDA_TRY(cudaEventRecord(s.ev0, stream));
        CUDA_TRY(small_sweep_launch(p->pd[di].dp, b, stream));
        if (prof) CUDA_TRY(cudaEventRecord(s.ev1, stream));
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
    if (prof && p->small_path) {
        float ms = 0;
        CUDA_TRY(cudaEventElapsedTime(&ms, s.ev0, s.ev1));
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
        cudaStreamSynchronize(s.stream);
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
    st.path = (p && !p->small_path) ? 1 : 0;
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
    cudaStream_t st = s.stream;
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
    if (prof) CUDA_TRY(cudaEventRecord(s.ev0, st));
    CUDA_TRY(small_fit_launch(p->pd[di].dp, fp, fb, st));
    if (prof) CUDA_TRY(cudaEventRecord(s.ev1, st));
    CUDA_TRY(cudaMemcpyAsync(s.fit_ll.h, s.fit_ll.d, (size_t)m * sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(s.fit_theta.h, s.fit_theta.d, (size_t)m * n * sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(s.fit_iters.h, s.fit_iters.d, (size_t)m * sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(s.fit_nfev.h, s.fit_nfev.d, (size_t)m * sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(s.fit_status.h, s.fit_status.d, (size_t)m * sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(s.fit_counters.h, s.fit_counters.d, 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (prof) {
        float ms = 0;
        CUDA_TRY(cudaEventElapsedTime(&ms, s.ev0, s.ev1));
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
    if (p->small_path && (!host_loop || o.optimizer == GPCC_OPT_NELDERMEAD)) return fit_shard_device(p, di, idx, delays, P, theta0, o, out);
    if (o.optimizer == GPCC_OPT_NELDERMEAD)
        return fail(-7, "the Nelder-Mead option runs on the fused small-N path only (N <= 199); use the default L-BFGS");
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
    if (!p->small_path && o.max_iter <= 0 && !o.theta0_per_candidate && L >= 2) {
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

int gpcc_version(void) { return 101; }   // 101: gpcc_stats grew by n_tau_cache and assembly_bytes (appended)
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
    gpcc_ctx* ctx = new gpcc_ctx();
    ctx->ds.resize(ndev);
    for (int i = 0; i < ndev; ++i) {
        DeviceState& s = ctx->ds[i];
        s.dev = dev_ids ? dev_ids[i] : i;
        if (s.dev < 0 || s.dev >= count) { delete ctx; return fail(-3, "invalid device id"); }
        cudaDeviceProp prop;
        CUDA_TRY(cudaGetDeviceProperties(&prop, s.dev));
        if (prop.major < 10) { delete ctx; return fail(-4, "libgpcc_b200 is built for sm_100a (Blackwell B200) only"); }
        CUDA_TRY(cudaSetDevice(s.dev));
        // highest priority: in the tiled path this stream carries the critical pivot/panel chain while the bulk of each
        // trailing update runs on a low-priority stream (large_path.cu), so pivot CTAs get the next free SM
        int prio_lo = 0, prio_hi = 0;
        CUDA_TRY(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
        CUDA_TRY(cudaStreamCreateWithPriority(&s.stream, cudaStreamNonBlocking, prio_hi));
        CUDA_TRY(cudaEventCreate(&s.ev0));
        CUDA_TRY(cudaEventCreate(&s.ev1));
    }
    *out = ctx;
    return 0;
}

int gpcc_ctx_destroy(gpcc_ctx* ctx) {
    if (!ctx) return 0;
    if (ctx->nccl) nccl_bridge_destroy(ctx->nccl);
    for (auto& s : ctx->ds) {
        cudaSetDevice(s.dev);
        EvalSlot& q = s.slot;
        q.delays.release(); q.alpha.release(); q.rho.release(); q.ll.release(); q.grad.release(); q.info.release();
        s.post_ll.release(); s.post_prior.release(); s.post_out.release();
        s.gat_send.release(); s.gat_recv.release(); s.gat_post.release();
        s.fit_delays.release(); s.fit_theta0.release(); s.fit_ll.release(); s.fit_theta.release();
        s.fit_iters.release(); s.fit_nfev.release(); s.fit_status.release(); s.fit_counters.release(); s.fit_order.release();
        if (s.ev0) cudaEventDestroy(s.ev0);
        if (s.ev1) cudaEventDestroy(s.ev1);
        large_workspace_release(s.large);
        if (s.stream) cudaStreamDestroy(s.stream);
    }
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
    gpcc_problem* p = new gpcc_problem();
    p->ctx = ctx; p->L = L; p->kernel_id = kernel_id;
    p->n_per_band.assign(n_per_band, n_per_band + L);
    p->band_start.assign(L + 1, 0);
    for (int l = 0; l < L; ++l) {
        if (n_per_band[l] < 1) { delete p; return fail(-4, "every band needs at least one observation"); }
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
        if (!(p->Sigmab[l] > 0) || !std::isfinite(p->mub[l])) {
            delete p;
            return fail(-5, "prior of the shift b is degenerate (band with <2 points or zero variance)");
        }
    }
    p->band.resize(N); p->resid.resize(N); p->s2.resize(N); p->sigb.resize(N);
    for (int l = 0; l < L; ++l)
        for (int i = p->band_start[l]; i < p->band_start[l + 1]; ++i) {
            p->band[i] = l;
            p->resid[i] = y[i] - p->mub[l];              // Y - Q*mu_b (:98, :139)
            p->s2[i] = sigma[i] * sigma[i];              // Sobs (:89)
            p->sigb[i] = p->Sigmab[l];                   // B = Q Sigma_b Q' (:96)
            if (!std::isfinite(t[i]) || !std::isfinite(y[i]) || !std::isfinite(sigma[i])) {
                delete p;
                return fail(-6, "non-finite input data");
            }
        }
    p->small_path = small_path_supports(N);
    p->pd.resize(ctx->ds.size());
    struct Guard { gpcc_problem* p; ~Guard() { if (p) gpcc_problem_destroy(p); } } guard{p};   // a failed upload frees what exists
    for (size_t di = 0; di < ctx->ds.size(); ++di) {
        auto& d = p->pd[di];
        d.dev = ctx->ds[di].dev;
        CUDA_TRY(cudaSetDevice(d.dev));
        CUDA_TRY(cudaMalloc(&d.t, N * sizeof(double)));
        CUDA_TRY(cudaMalloc(&d.resid, N * sizeof(double)));
        CUDA_TRY(cudaMalloc(&d.y, N * sizeof(double)));
        CUDA_TRY(cudaMalloc(&d.s2, N * sizeof(double)));
        CUDA_TRY(cudaMalloc(&d.sigb, N * sizeof(double)));
        CUDA_TRY(cudaMalloc(&d.band, N * sizeof(int)));
        CUDA_TRY(cudaMemcpy(d.t, p->t.data(), N * sizeof(double), cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMemcpy(d.resid, p->resid.data(), N * sizeof(double), cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMemcpy(d.y, p->y.data(), N * sizeof(double), cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMemcpy(d.s2, p->s2.data(), N * sizeof(double), cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMemcpy(d.sigb, p->sigb.data(), N * sizeof(double), cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMemcpy(d.band, p->band.data(), N * sizeof(int), cudaMemcpyHostToDevice));
        d.dp.N = N; d.dp.L = L; d.dp.kernel_id = kernel_id;
        d.dp.t = d.t; d.dp.resid = d.resid; d.dp.y = d.y; d.dp.s2 = d.s2; d.dp.sigb = d.sigb; d.dp.band = d.band;
        for (int l = 0; l <= L; ++l) d.dp.band_start[l] = p->band_start[l];
    }
    guard.p = nullptr;
    *out = p;
    return 0;
}

int gpcc_problem_destroy(gpcc_problem* p) {
    if (!p) return 0;
    if (p->cached_state) { gpcc_fit_state_destroy(p->cached_state); p->cached_state = nullptr; }
    // only the problem's own copies of the device ids are read here: the context may already be gone (finalizer order in
    // Julia / Python is unspecified), see the lifetime rule in include/gpcc_b200.h
    for (size_t di = 0; di < p->pd.size(); ++di) {
        auto& d = p->pd[di];
        cudaSetDevice(d.dev);
        cudaFree(d.t); cudaFree(d.resid); cudaFree(d.y); cudaFree(d.s2); cudaFree(d.sigb); cudaFree(d.band);
    }
    delete p;
    return 0;
}

int gpcc_problem_get_prior(const gpcc_problem* p, double* mub, double* Sigmab) {
    if (!p) return fail(-1, "problem is NULL");
    if (mub) std::memcpy(mub, p->mub.data(), p->L * sizeof(double));
    if (Sigmab) std::memcpy(Sigmab, p->Sigmab.data(), p->L * sizeof(double));
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
        if (!p->small_path && !want_grad && !theta && L >= 2) {
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
    // persistent buffers: cudaMalloc/cudaFree serialise against every other context on the box (and stall for hundreds
    // of milliseconds when several ranks with NCCL peer mappings hit them at once), so the hot path never calls them
    CUDA_TRY(s.post_ll.reserve(M));
    CUDA_TRY(s.post_out.reserve(M));
    if (logprior) CUDA_TRY(s.post_prior.reserve(M));
    std::memcpy(s.post_ll.h, loglik, (size_t)M * sizeof(double));
    CUDA_TRY(cudaMemcpyAsync(s.post_ll.d, s.post_ll.h, (size_t)M * sizeof(double), cudaMemcpyHostToDevice, s.stream));
    if (logprior) {
        std::memcpy(s.post_prior.h, logprior, (size_t)M * sizeof(double));
        CUDA_TRY(cudaMemcpyAsync(s.post_prior.d, s.post_prior.h, (size_t)M * sizeof(double), cudaMemcpyHostToDevice, s.stream));
    }
    CUDA_TRY(posterior_launch(M, s.post_ll.d, logprior ? s.post_prior.d : nullptr, s.post_out.d, s.stream));
    CUDA_TRY(cudaMemcpyAsync(s.post_out.h, s.post_out.d, (size_t)M * sizeof(double), cudaMemcpyDeviceToHost, s.stream));
    CUDA_TRY(cudaStreamSynchronize(s.stream));
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
        CUDA_TRY(cudaMemcpyAsync(s.gat_send.d, h, (size_t)per * REC * sizeof(double), cudaMemcpyHostToDevice, s.stream));
        CUDA_TRY(posterior_partial_launch(per, REC, JCOL, s.gat_send.d, s.stream));
        d_send[di] = s.gat_send.d; d_recv[di] = s.gat_recv.d; streams[di] = s.stream;
    }
    std::string err;
    if (nccl_bridge_allgather(ctx->nccl, d_send, d_recv, (int)blk, streams, err)) return fail(2001, "ncclAllGather: " + err);
    DeviceState& s0 = ctx->ds[0];
    CUDA_TRY(cudaSetDevice(s0.dev));
    CUDA_TRY(s0.gat_post.reserve((size_t)per * G));
    CUDA_TRY(posterior_combine_launch(G, per, REC, JCOL, s0.gat_recv.d, s0.gat_post.d, s0.stream));
    CUDA_TRY(cudaMemcpyAsync(s0.gat_post.h, s0.gat_post.d, (size_t)per * G * sizeof(double), cudaMemcpyDeviceToHost, s0.stream));
    CUDA_TRY(cudaMemcpyAsync(s0.gat_recv.h, s0.gat_recv.d, blk * G * sizeof(double), cudaMemcpyDeviceToHost, s0.stream));
    CUDA_TRY(cudaStreamSynchronize(s0.stream));
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
