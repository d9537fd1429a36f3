/*
 * gpcc_b200.h -- C ABI of the B200-native (sm_100a) replacement for the GPCC.jl hot path.
 *
 * The reference (HITS-AIN/GPCC.jl v0.1.35) is pure Julia and has no FFI; this header is the contract a
 * thin Julia `ccall` shim (julia/GPCC_B200.jl, INTEGRATION.md) binds instead of the reference's Julia
 * functions.  Each entry cites the reference code it replaces (paths relative to /root/reference).
 *
 * Conventions
 *   - plain C, all floating point is FP64, all arrays are caller-owned contiguous HOST memory;
 *     per-band data are concatenated in band order (Julia `reduce(vcat, ...)`); matrices are
 *     column-major (Julia layout).  The library never keeps a caller pointer after returning.
 *   - every function returns 0 on success, <0 for an invalid argument, >0 for a CUDA/NCCL failure;
 *     gpcc_last_error() gives the text.  Numerical failure (matrix not positive definite) is reported
 *     per element in `info` (LAPACK convention: k>0 = leading minor k not PD) with loglik = -Inf; it is
 *     never a return code.  No exception, exit or signal crosses the boundary.
 *   - calls are synchronous; a context is not thread-safe.
 *   - there is NO CPU fallback: without a CUDA device gpcc_ctx_create fails.
 *   - lifetime: a problem and a fit state may only be USED while their context (and, for a fit state, its problem)
 *     is alive; they may be DESTROYED in any order, also after the context (garbage-collected hosts run
 *     finalizers in unspecified order): destroy functions only touch memory the object itself owns.
 */
#ifndef GPCC_B200_H
#define GPCC_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define GPCC_MAX_BANDS 8

/* src/util.jl:15-52 -- the four scalar kernels; the Julia shim maps function identity to this enum. */
enum { GPCC_KERNEL_OU = 0, GPCC_KERNEL_RBF = 1, GPCC_KERNEL_MATERN32 = 2, GPCC_KERNEL_MATERN52 = 3 };

/* Parameter transforms of src/gpccfixdelay_marginaliseb.jl:112-114 (MiscUtil.makepositive /
 * transformbetween, un-vendored): id 0 = softplus + 1e-8 floor, rhomin+(rhomax-rhomin)*logistic.   */
enum { GPCC_TRANSFORM_SOFTPLUS_LOGISTIC = 0 };
enum { GPCC_OPT_LBFGS = 0, GPCC_OPT_NELDERMEAD = 1 };
/* How a problem evaluates its likelihood: the dense factorisation of K + Sobs + B (default), or an exact Kalman filter
 * over the merged, delay-shifted times (OU, matern32, matern52 only; see gpcc_problem_set_method).                  */
enum { GPCC_METHOD_DENSE = 0, GPCC_METHOD_STATESPACE = 1 };

typedef struct gpcc_ctx gpcc_ctx;
typedef struct gpcc_problem gpcc_problem;
typedef struct gpcc_fit_state gpcc_fit_state;
typedef struct gpcc_ss_state gpcc_ss_state;

/* Keyword arguments / constants of gpcc (src/gpccfixdelay_marginaliseb.jl:46, :69, :112, :205). */
typedef struct gpcc_fit_options {
    int    max_iter;        /* `iterations`: cap on optimiser iterations per candidate            */
    double rhomin;          /* `rhomin` (default 0.1)                                              */
    double rhomax;          /* `rhomax`                                                            */
    double alpha_floor;     /* 1e-8  (:112)                                                        */
    double gtol;            /* stop when max|d(-logL)/dtheta| <= gtol   (L-BFGS; default 1e-7)      */
    double ftol;            /* stop when the relative decrease of -logL <= ftol twice (1e-13)      */
    int    history;         /* L-BFGS memory (default 8, max 16)                                   */
    int    transform_id;    /* GPCC_TRANSFORM_*                                                    */
    int    theta0_per_candidate; /* 0: theta0 is [P][L+1] shared by all candidates (the reference's
                                    seed=1 behaviour, :62); 1: theta0 is [M][P][L+1]               */
    int    optimizer;       /* GPCC_OPT_LBFGS (default) or GPCC_OPT_NELDERMEAD: the reference's own optimiser
                               (:205-211, g_tol = nm_gtol), on the device, for basin-for-basin comparisons;
                               fused small-N path only (N <= 199)                                  */
    double nm_gtol;         /* Optim.Options(g_tol = 1e-6) (:205): simplex spread at which Nelder-Mead stops */
} gpcc_fit_options;

/* Per-stage device timings of the most recent call, measured with CUDA events on the library's own
 * streams (only when enabled with gpcc_ctx_set_profiling).                                          */
typedef struct gpcc_stats {
    double ms_total;            /* whole call, host wall clock                                      */
    double ms_eval_kernels;     /* sum of likelihood(+gradient) kernel time, CUDA events            */
    double ms_assembly;         /* large-N path: covariance assembly kernels                        */
    double ms_factor;           /* large-N path: pivot + panel + trailing-update kernels            */
    double ms_gradreduce;       /* large-N path: gradient reduction kernel                          */
    long long n_eval_launches;  /* kernels launched by this library in the call                     */
    long long n_evals;          /* (candidate, theta) evaluations                                   */
    long long n_evals_grad;     /* ... of which with gradient                                       */
    int    path;                /* 0 = fused register-resident small-N kernel, 1 = tiled large-N,
                                   2 = state-space method (Kalman filter, gpcc_problem_set_method)   */
    int    n_devices;
    long long n_shared_prefix;  /* tiled path, logL only: evaluations whose leading block (all bands but the
                                   last) was factorised by another evaluation of their wave (structure reuse) */
    long long n_tau_cache;      /* tiled path, fixed-theta sweep over >= 3 bands: evaluations that took the band-1 steps of
                                   their last band (a function of the last delay alone) from the last-band cache            */
    long long assembly_bytes;   /* tiled path: HBM bytes the assembly kernels of the busiest device moved (tiles written;
                                   tiles imported from the last-band cache count read + written); pairs with ms_assembly      */
} gpcc_stats;

int         gpcc_version(void);   /* 103.  102 -> 103: gpcc_ss_state_* (additive); gpcc_ss_sample and gpcc_ss_state_sample were
                                      added later under the same number (additive: a caller that needs one looks the symbol up).  101 -> 102: gpcc_problem_set_method (additive).
                                      100 -> 101: gpcc_stats grew by n_tau_cache and assembly_bytes (appended at the end);
                                      a caller built against 100 must be rebuilt before it calls gpcc_ctx_get_stats                */
const char* gpcc_last_error(void);

/* CUDA contexts, streams, workspaces on `ndev` devices (dev_ids NULL = 0..ndev-1).  With ndev>1 the
 * candidate grid is sharded over the devices (README.md:185-206 `pmap`) and the per-candidate
 * log-likelihoods are combined with one NCCL allgather.                                             */
int gpcc_ctx_create(int ndev, const int* dev_ids, gpcc_ctx** out);
int gpcc_ctx_destroy(gpcc_ctx* ctx);
/* One process per GPU (torchrun; one Julia `Distributed` worker per device, README.md:185-189): rank 0 draws an id,
 * the host program hands its 128 bytes to every rank, and each rank attaches its ONE-device context.  From then on
 * gpcc_fit_batch fits only the candidates m with m mod world == rank, and gpcc_grid_posterior (called by EVERY rank with
 * the same arguments) all-gathers the per-candidate records over NCCL and returns the full outputs on every rank.   */
int gpcc_comm_unique_id(char* out_id128);
int gpcc_ctx_comm_init_rank(gpcc_ctx* ctx, int world, int rank, const char* id128);
int gpcc_ctx_set_profiling(gpcc_ctx* ctx, int enabled);
int gpcc_ctx_get_stats(const gpcc_ctx* ctx, gpcc_stats* out);
int gpcc_ctx_device_count(const gpcc_ctx* ctx);

/* Data of one gpcc call (src/gpccfixdelay_marginaliseb.jl:85-98): L bands, n_per_band[l] points each,
 * t / y / sigma concatenated (N = sum n).  mub / Sigmab (length L: prior mean and the *diagonal* of the
 * inflated prior covariance, :92-94) may be NULL, in which case the library computes mean(y_l) and
 * 100*var(y_l) (unbiased) itself.  The data are uploaded to every device of the context.            */
int gpcc_problem_create(gpcc_ctx* ctx, int L, const int* n_per_band, const double* t, const double* y,
                        const double* sigma, int kernel_id, const double* mub, const double* Sigmab,
                        gpcc_problem** out);
int gpcc_problem_destroy(gpcc_problem* p);
int gpcc_problem_get_prior(const gpcc_problem* p, double* mub, double* Sigmab);

/* Select how the problem evaluates its likelihood; a problem starts in GPCC_METHOD_DENSE and may switch back and forth.
 * GPCC_METHOD_STATESPACE (OU, matern32, matern52; rbf has no finite state-space form and is rejected) computes the same
 * logL, gradient and postb exactly, by a Kalman filter over the N merged, delay-shifted times: O(N (d+L)^2) per
 * evaluation (d = 1, 2, 3) instead of the N^3/3 of the dense factorisation, and O(N) memory.  Switching it on sorts
 * every band by time once and uploads that copy to every device.  Under it:
 *   - gpcc_loglik_batch / gpcc_loglik_theta_batch run the filter; info > 0 is the 1-based position, in the merged
 *     order of the shifted times (ties to the lower band), of the first observation whose innovation variance is not
 *     positive and finite (loglik = -Inf).  It is a position in that order, not a leading-minor index;
 *   - gpcc_fit_batch / gpcc_grid_posterior always use the host-driven batched L-BFGS (screening, then one batched
 *     evaluation per round), whatever N is; GPCC_OPT_NELDERMEAD is rejected with -7;
 *   - gpcc_postb runs one filter and returns its final b-block;
 *   - gpcc_fit_state_*, gpcc_predict, gpcc_predict_loglik and gpcc_fit_state_sample stay dense: a fit state is a
 *     Cholesky factor of K + Sobs;
 *   - gpcc_ss_state_create builds the O(N) fit state of this method (see below): predictive means, standard deviations
 *     and the test log-likelihood without a factorisation;
 *   - gpcc_ss_sample draws from N(0, K + Sobs) in O(N), the O(N) form of gpcc_fit_state_sample;
 *   - gpcc_ss_state_sample draws the test values jointly from the predictive distribution N(mu_pred, Sigma_pred) in
 *     O(N + NT) per draw.
 * The full predictive covariance has no O(N) form and stays dense; its joint draws do not need it.
 * Returns < 0 for a NULL problem, an unknown method, or rbf with GPCC_METHOD_STATESPACE.                              */
int gpcc_problem_set_method(gpcc_problem* p, int method);

/* objective(alpha, rho) of src/gpccfixdelay_marginaliseb.jl:133-141 for M (delay, hyper-parameter)
 * pairs in constrained space: K~ = delayedCovariance (src/delayedCovariance.jl:1-38) + Sobs + B,
 * logpdf(MvNormal(bbar, K~), Y).  want_grad adds d logL / d(alpha_1..alpha_L, rho) (not in the
 * reference, which is derivative free).  delays, alpha: [M][L]; rho, out_ll: [M];
 * out_grad: [M][L+1] (may be NULL when want_grad == 0); out_info: [M] (may be NULL).                */
int gpcc_loglik_batch(gpcc_problem* p, int M, const double* delays, const double* alpha, const double* rho,
                      int want_grad, double* out_ll, double* out_grad, int* out_info);

/* Same objective in the optimiser's unconstrained parameters theta = [L+1] (unpack, :116-126), with
 * the gradient chained through the transforms.                                                      */
int gpcc_loglik_theta_batch(gpcc_problem* p, int M, const double* delays, const double* theta,
                            const gpcc_fit_options* opt, int want_grad, double* out_ll, double* out_grad,
                            int* out_info);

/* getsolution (src/gpccfixdelay_marginaliseb.jl:203-215) for M candidate delay vectors at once:
 * stage 1 evaluates the P (`initialrandom`) start points theta0 and keeps the best (:207-209); stage 2
 * maximises logL from there (:211; host-driven batched L-BFGS with the analytic gradient instead of
 * Nelder-Mead).  Outputs (any may be NULL): out_ll[M] = -result.minimum (:351), out_theta[M][L+1],
 * out_alpha[M][L], out_rho[M], out_iters[M], out_nfev[M], out_info[M] (0 converged, 1 iteration cap,
 * 2 line search stalled, <0 no start point was positive definite).                                  */
int gpcc_fit_batch(gpcc_problem* p, int M, const double* delays, int P, const double* theta0,
                   const gpcc_fit_options* opt, double* out_ll, double* out_theta, double* out_alpha,
                   double* out_rho, int* out_iters, int* out_nfev, int* out_info);

/* The README's grid driver (README.md:170-178, 185-210, 285) followed by getprobabilities
 * (src/getprobabilities.jl:1-20): fit every candidate (sharded over the context's devices, candidate
 * m on device m mod ndev), allgather the log-likelihoods, normalise with log-sum-exp under `logprior`
 * (NULL = flat).  out_post[M] sums to 1; the other outputs are as in gpcc_fit_batch.                */
int gpcc_grid_posterior(gpcc_problem* p, int M, const double* delays, const double* logprior, int P,
                        const double* theta0, const gpcc_fit_options* opt, double* out_ll, double* out_post,
                        double* out_theta, double* out_alpha, double* out_rho, int* out_nfev, int* out_info);

/* src/getprobabilities.jl:10-20 on the device: exp(ll + logprior - logsumexp(ll + logprior));
 * logprior NULL = the 1-argument method (:1-6).                                                     */
int gpcc_getprobabilities(gpcc_ctx* ctx, int M, const double* loglik, const double* logprior, double* out_post);

/* What the reference's `pred` closures capture after the fit (src/gpccfixdelay_marginaliseb.jl:235-252: alpha, rho,
 * KSobsB, postb): ONE Cholesky factorisation of K + Sobs at the fitted (delays, alpha, rho), kept on the device
 * together with postb, and reused by every later prediction (the reference re-factorises on each call, :275, :283).
 * Returns -6 when K + Sobs is not positive definite.                                                   */
int gpcc_fit_state_create(gpcc_problem* p, const double* delays, const double* alpha, double rho, gpcc_fit_state** out);
int gpcc_fit_state_destroy(gpcc_fit_state* s);
/* postb (:248-252): out_mu[L], out_Sigma[L*L] (symmetrised, :252).                                     */
int gpcc_fit_state_postb(const gpcc_fit_state* s, double* out_mu, double* out_Sigma);
/* predictTest (:259-307) and the test log-likelihood (:311-343) from the cached factor; arguments as in
 * gpcc_predict / gpcc_predict_loglik below.                                                            */
int gpcc_fit_state_predict(gpcc_fit_state* s, const int* ntest_per_band, const double* ttest, double* out_mu,
                           double* out_sd, double* out_Sigma);
int gpcc_fit_state_predict_loglik(gpcc_fit_state* s, const int* ntest_per_band, const double* ttest,
                                  const double* ytest, const double* sigmatest, double* out_ll, int* out_info);
/* Draws from the process at the state's hyper-parameters, on the device: out_f[s][N] = Lc z_s with Lc Lc' = K + Sobs and
 * z_s ~ N(0, I) from a counter-based generator (Philox-4x32-10 + Box-Muller, reproducible per seed).  This is the sampling
 * step of the reference's simulator (src/simulatedata.jl:128-145: Y ~ MvNormal(0, C), C = delayedCovariance(OU, ...)) for
 * large synthetic benchmarks (SURVEY 8f-4); the light curves around it (scaling, offsets, noise: :151-159) are O(N) host
 * arithmetic in both shims.  out_z (may be NULL) receives the deviates [nsamples][N].                                  */
int gpcc_fit_state_sample(gpcc_fit_state* s, unsigned long long seed, int nsamples, double* out_f, double* out_z);
/* diagnostics: number of N^3 factorisations this state has run (1 for its whole life).               */
long long gpcc_fit_state_factorisations(const gpcc_fit_state* s);

/* Stateless forms of the three calls above.  They keep the fit state of the most recent (delays, alpha, rho) on
 * the problem, so postb + any number of pred calls at the fitted hyper-parameters share one factorisation.
 * Posterior of the shifts b (src/gpccfixdelay_marginaliseb.jl:248-252): out_mu[L], out_Sigma[L*L].  */
int gpcc_postb(gpcc_problem* p, const double* delays, const double* alpha, double rho, double* out_mu,
               double* out_Sigma);

/* predictTest (src/gpccfixdelay_marginaliseb.jl:259-307).  ttest holds ntest_per_band[l] times per band,
 * concatenated (NT = sum).  out_mu[NT]; out_sd[NT] = sqrt(max(diag(Sigma_pred), 1e-6)) (:303) if not
 * NULL; out_Sigma[NT*NT] = full predictive covariance incl. the 1e-8 jitter (:279) if not NULL.      */
int gpcc_predict(gpcc_problem* p, const double* delays, const double* alpha, double rho,
                 const int* ntest_per_band, const double* ttest, double* out_mu, double* out_sd,
                 double* out_Sigma);

/* pred(ttest, ytest, sigmatest) (src/gpccfixdelay_marginaliseb.jl:311-343): test log-likelihood under
 * N(mu_pred, Sigma_pred + diag(sigmatest^2)); out_info = 0, or k>0 if that matrix is not PD (the
 * reference then repairs it with MiscUtil.nearestposdef on the host, which the caller keeps doing).  */
int gpcc_predict_loglik(gpcc_problem* p, const double* delays, const double* alpha, double rho,
                        const int* ntest_per_band, const double* ttest, const double* ytest,
                        const double* sigmatest, double* out_ll, int* out_info);

/* Fit state of the state-space method (a problem in GPCC_METHOD_STATESPACE; OU, matern32, matern52) at (delays, alpha, rho):
 * one forward Kalman filter that stores its filtered moments and one backward (Bryson-Frazier) pass over the N merged
 * training points, on the problem's first device.  O(N (d+L)^2) memory and time, no N x N matrix.  The state owns all it
 * reads (its own copy of the sorted training data, mu_b, Sigma_b and ll(train)): it may be used after its problem is
 * destroyed or switched back to GPCC_METHOD_DENSE.  Returns < 0 for a NULL argument, a problem not in
 * GPCC_METHOD_STATESPACE, alpha <= 0, rho <= 0 or non-finite values; -6 when the filter meets an innovation variance
 * that is not positive and finite.                                                                                      */
int gpcc_ss_state_create(gpcc_problem* p, const double* delays, const double* alpha, double rho, gpcc_ss_state** out);
int gpcc_ss_state_destroy(gpcc_ss_state* s);
/* Per-point predictTest (:293-307): out_mu[NT] and out_sd[NT] (may be NULL) as gpcc_fit_state_predict returns them (sd =
 * sqrt(max(var + 1e-8, 1e-6))), in O((d+L)^3) per test point; test times in any order.  The full predictive covariance
 * needs the dense fit state.  Returns < 0 for negative counts or non-finite times; NT = 0 does nothing.             */
int gpcc_ss_state_predict(gpcc_ss_state* s, const int* ntest_per_band, const double* ttest, double* out_mu, double* out_sd);
/* Test log-likelihood (:311-343), logpdf(N(mu_pred, Sigma_pred + diag(sigmatest^2)), ytest) with the 1e-8 jitter in
 * Sigma_pred, as ll(train + test) - ll(train): one filter over the N + NT merged points.  out_info (may be NULL) = 0, or the
 * 1-based merged position of the first innovation variance that is not positive and finite (out_ll = -Inf).  Returns < 0
 * for negative counts, non-finite times or values, or sigmatest < 0; NT = 0 gives out_ll = 0.                         */
int gpcc_ss_state_predict_loglik(gpcc_ss_state* s, const int* ntest_per_band, const double* ttest, const double* ytest,
                                 const double* sigmatest, double* out_ll, int* out_info);
/* Exact joint draws of the test values g*_j = alpha_l f(t*_j - tau_l) + b_l + eta_j (eta_j ~ N(0, 1e-8), the jitter) given
 * the training data: out_f[nsamples][NT] ~ N(mu_pred, Sigma_pred) of pred(::Vector{Vector}) (:259-289), test points in the
 * order of ttest (bands concatenated, any order within a band), in O(N + NT) time and memory per draw and no N x N or
 * NT x NT matrix.  Pathwise conditioning: a joint prior draw over the N training and NT test times (the recurrence of
 * gpcc_ss_sample over their merge) and of the shifts, corrected by the smoother mean of the residual of that draw with the
 * state's own gains.  Deviates, one array [nsamples][N+NT][d+1] then [nsamples][L]: per sample the d process deviates and the
 * noise deviate of every point (the training points in the problem's input order, then the test points in the order of
 * ttest), then the L shift deviates (b_l = mu_b,l + sqrt(Sigma_b,l) zeta_l in the prior draw).  z_in (may be NULL) supplies
 * them, and seed is then ignored; otherwise they come from Philox-4x32-10 + Box-Muller in a stream of their own and depend
 * only on (seed, sample, slot), so a draw does not depend on nsamples.  out_z (may be NULL) receives the deviates used.
 * Bitwise reproducible.  Returns -1 for a NULL argument, -3 for a non-finite test time, -5 for a negative count, -7 for
 * nsamples < 1 or too many points, -8 for a non-finite value in z_in; NT = 0 writes nothing.                            */
int gpcc_ss_state_sample(gpcc_ss_state* s, const int* ntest_per_band, const double* ttest, unsigned long long seed,
                         int nsamples, const double* z_in, double* out_f, double* out_z);

/* Exact draws f ~ N(0, K + Sobs) at (delays, alpha, rho) for a problem in GPCC_METHOD_STATESPACE, the distribution of
 * gpcc_fit_state_sample, in O(N) time and memory: the kernel's SDE recurrence over the merged, delay-shifted times, run as a
 * parallel scan on the problem's first device.  out_f[nsamples][N] is in the problem's input order.  Deviates: d process
 * deviates then 1 noise deviate per point (d = 1, 2, 3 for OU, matern32, matern52), [nsamples][N][d+1]; the d process
 * deviates of point i drive the step of the recurrence that arrives at i.  z_in (may be NULL) supplies them, and seed is
 * then ignored; otherwise they come from Philox-4x32-10 + Box-Muller and depend only on (seed, sample, point), so a draw
 * does not depend on nsamples and the same seed gives common random numbers across delays.  out_z (may be NULL) receives
 * the deviates used.  Bitwise reproducible.  Returns < 0 as gpcc_ss_state_create does (-1 NULL, -2 alpha <= 0, -3
 * non-finite delay, -4 rho <= 0, -5 problem not in GPCC_METHOD_STATESPACE), -7 for nsamples < 1 and -8 for a non-finite
 * value in z_in.                                                                                                        */
int gpcc_ss_sample(gpcc_problem* p, const double* delays, const double* alpha, double rho, unsigned long long seed,
                   int nsamples, const double* z_in, double* out_f, double* out_z);

/* Fill `opt` with the reference defaults (seed-independent part of :46, :112, :205).               */
int gpcc_fit_options_default(gpcc_fit_options* opt);

#ifdef __cplusplus
}
#endif
#endif /* GPCC_B200_H */
