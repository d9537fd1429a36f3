// Batched L-BFGS: one small state machine per delay candidate.  Replaces the per-candidate
// optimize(..., NelderMead(), ...) of /root/reference/src/gpccfixdelay_marginaliseb.jl:205-211
// as north_star specifies.  Minimises f = -logL over the unconstrained theta in R^(L+1).
// The same code runs in two drivers:
//   * on the DEVICE (small_fit.cu): one persistent CTA per candidate keeps this state in shared memory and alternates
//     evaluation and update without leaving the kernel (fused small-N path, the default);
//   * on the host (api.cu, fit_shard): every round gathers the trial points of all active candidates into ONE batched
//     device evaluation and feeds the results back (tiled large-N path, where one evaluation is many kernels).
#pragma once
#include <cmath>

#if defined(__CUDACC__)
#define GPCC_HD __host__ __device__
#else
#define GPCC_HD
#endif

namespace gpcc {

GPCC_HD inline bool lb_finite(double x) { return x - x == 0.0; }          // false for +-Inf and NaN
GPCC_HD inline double lb_inf() { return __builtin_huge_val(); }
GPCC_HD inline void lb_copy(double* dst, const double* src, int n) { for (int i = 0; i < n; ++i) dst[i] = src[i]; }

constexpr int LBFGS_MAXN = 9;    // L+1 <= GPCC_MAX_BANDS+1
constexpr int LBFGS_MAXM = 16;
constexpr double STEP_CAP = 2.0;   // max |delta theta_i| per L-BFGS iteration

struct LbfgsOptions {
    int max_iter = 1000;
    double gtol = 1e-7;
    double ftol = 1e-13;
    int history = 8;
    int max_ls = 30;
    int n_scale = 0;        // the first n_scale coordinates are softplus scales (alpha): their step cap grows with the coordinate
    double rel_cap = 0.25;  // ... to rel_cap * theta_i once that exceeds STEP_CAP
};

struct LbfgsState {
    enum Status { RUNNING = -100, CONVERGED = 0, ITER_CAP = 1, LS_STALL = 2, NO_START = -1 };
    int n = 0;
    int status = RUNNING;
    int iters = 0, nfev = 0;
    double x[LBFGS_MAXN], g[LBFGS_MAXN], f = 0.0;
    double d[LBFGS_MAXN], xt[LBFGS_MAXN];
    double t = 1.0, tlo = 0.0, thi = 0.0, gd0 = 0.0, tcap = 0.0;
    int ls_trials = 0;
    bool have_fb = false;              // best Armijo point seen in this line search (fallback)
    double fb_x[LBFGS_MAXN], fb_g[LBFGS_MAXN], fb_f = 0.0;
    double S[LBFGS_MAXM][LBFGS_MAXN], Y[LBFGS_MAXM][LBFGS_MAXN], R[LBFGS_MAXM];
    int hcount = 0, hhead = 0;         // ring buffer
    int small_df = 0;
    int n_scale = 0;                   // copies of the options new_direction needs
    double rel_cap = 0.0;

    GPCC_HD static double dot(const double* a, const double* b, int n) {
        double s = 0.0;
        for (int i = 0; i < n; ++i) s += a[i] * b[i];
        return s;
    }

    GPCC_HD void start(int n_, const double* x0, double f0, const double* g0, const LbfgsOptions& o) {
        n = n_;
        lb_copy(x, x0, n);
        lb_copy(g, g0, n);
        f = f0;
        status = RUNNING;
        iters = 0;
        hcount = hhead = 0;
        small_df = 0;
        n_scale = o.n_scale;
        rel_cap = o.rel_cap;
        double gmax = 0.0;
        for (int i = 0; i < n; ++i) gmax = fmax(gmax, fabs(g[i]));
        if (!(gmax > o.gtol)) { status = CONVERGED; return; }
        if (o.max_iter <= 0) { status = ITER_CAP; return; }
        new_direction(true);
    }

    GPCC_HD void new_direction(bool first) {
        // two-loop recursion
        double qv[LBFGS_MAXN], a[LBFGS_MAXM];
        for (int i = 0; i < n; ++i) qv[i] = g[i];
        for (int k = 0; k < hcount; ++k) {
            const int idx = (hhead - 1 - k + 2 * LBFGS_MAXM) % LBFGS_MAXM;
            a[k] = R[idx] * dot(S[idx], qv, n);
            for (int i = 0; i < n; ++i) qv[i] -= a[k] * Y[idx][i];
        }
        if (hcount > 0) {
            const int idx = (hhead - 1 + LBFGS_MAXM) % LBFGS_MAXM;
            const double gamma = 1.0 / (R[idx] * dot(Y[idx], Y[idx], n));
            for (int i = 0; i < n; ++i) qv[i] *= gamma;
        }
        for (int k = hcount - 1; k >= 0; --k) {
            const int idx = (hhead - 1 - k + 2 * LBFGS_MAXM) % LBFGS_MAXM;
            const double bb = R[idx] * dot(Y[idx], qv, n);
            for (int i = 0; i < n; ++i) qv[i] += (a[k] - bb) * S[idx][i];
        }
        for (int i = 0; i < n; ++i) d[i] = -qv[i];
        gd0 = dot(g, d, n);
        if (!(gd0 < 0.0) || !lb_finite(gd0)) {     // not a descent direction: restart from steepest descent
            hcount = 0;
            for (int i = 0; i < n; ++i) d[i] = -g[i];
            gd0 = dot(g, d, n);
            first = true;
        }
        t = 1.0;
        if (first || hcount == 0) {
            const double gn = sqrt(dot(g, g, n));
            t = fmin(1.0, 1.0 / gn);
        }
        // Cap the step at STEP_CAP units of the unconstrained parameters per iteration.  theta lives on the softplus /
        // logistic scale: a jump of many units lands where the transforms saturate (alpha -> floor, rho -> rhomin), their
        // Jacobians vanish and a gradient method crawls for hundreds of iterations in a degenerate basin (SURVEY.md 7).
        // A scale far up the linear branch of the softplus (theta_i = alpha_i >> 1) is nowhere near saturation, and a fixed cap
        // makes the optimiser walk: the candidates at the edge of the grid, where the last band hardly overlaps the others,
        // have their optimum at alpha ~ 150 and needed 75 capped iterations to get there (the 170-220-evaluation tail of the
        // fitted grid).  For those coordinates the cap is rel_cap * theta_i once that exceeds STEP_CAP: geometric instead of
        // linear travel.  The rho coordinate (logistic) and everything at or below the knee keep the fixed cap.
        tcap = lb_inf();
        for (int i = 0; i < n; ++i) {
            const double ad = fabs(d[i]);
            if (!(ad > 0.0)) continue;
            const double cap = (i < n_scale) ? fmax(STEP_CAP, rel_cap * x[i]) : STEP_CAP;
            tcap = fmin(tcap, cap / ad);
        }
        t = fmin(t, tcap);
        tlo = 0.0;
        thi = lb_inf();
        ls_trials = 0;
        have_fb = false;
        for (int i = 0; i < n; ++i) xt[i] = x[i] + t * d[i];
    }

    GPCC_HD void accept(const double* xn, double fn, const double* gn, const LbfgsOptions& o, int hist) {
        double s[LBFGS_MAXN], y[LBFGS_MAXN];
        for (int i = 0; i < n; ++i) { s[i] = xn[i] - x[i]; y[i] = gn[i] - g[i]; }
        const double sy = dot(s, y, n);
        if (sy > 1e-10 * sqrt(dot(s, s, n) * dot(y, y, n)) && sy > 0.0) {
            lb_copy(S[hhead], s, n);
            lb_copy(Y[hhead], y, n);
            R[hhead] = 1.0 / sy;
            hhead = (hhead + 1) % LBFGS_MAXM;
            if (hcount < hist) ++hcount;
        }
        const double df = f - fn;
        lb_copy(x, xn, n);
        lb_copy(g, gn, n);
        f = fn;
        ++iters;
        double gmax = 0.0;
        for (int i = 0; i < n; ++i) gmax = fmax(gmax, fabs(g[i]));
        if (gmax <= o.gtol) { status = CONVERGED; return; }
        if (df <= o.ftol * fmax(1.0, fabs(f))) { if (++small_df >= 2) { status = CONVERGED; return; } }
        else small_df = 0;
        if (iters >= o.max_iter) { status = ITER_CAP; return; }
        new_direction(false);
    }

    // Feed the evaluation at xt (ok=false: matrix not PD / non-finite).  Afterwards either status != RUNNING
    // or xt holds the next trial point.
    GPCC_HD void feed(bool ok, double ft, const double* gt, const LbfgsOptions& o) {
        ++nfev;
        ++ls_trials;
        const int hist = o.history < 1 ? 1 : (o.history > LBFGS_MAXM ? LBFGS_MAXM : o.history);
        const double c1 = 1e-4, c2 = 0.9;
        bool armijo = ok && lb_finite(ft) && ft <= f + c1 * t * gd0;
        if (armijo) {
            const double gtd = dot(gt, d, n);
            if (gtd >= c2 * gd0) { accept(xt, ft, gt, o, hist); return; }   // weak Wolfe holds
            if ((thi == lb_inf()) && t >= tcap) { accept(xt, ft, gt, o, hist); return; }   // sufficient decrease at the step cap
            if (!have_fb || ft < fb_f) {
                have_fb = true; fb_f = ft;
                lb_copy(fb_x, xt, n);
                lb_copy(fb_g, gt, n);
            }
            tlo = t;
            t = (thi == lb_inf()) ? fmin(2.0 * t, tcap) : 0.5 * (tlo + thi);
        } else {
            // The objective carries ~1e-13 relative rounding noise.  Once the decrease the model predicts for this step is
            // below that noise, Armijo can no longer be verified and further backtracking only burns evaluations: the
            // point is converged to within the noise (remaining improvement <= |t g'd|, far below the 1e-6 target).
            const double noise = 4e-13 * fmax(1.0, fabs(f));
            if (ok && lb_finite(ft) && fabs(ft - f) <= noise && -t * gd0 <= noise) {
                if (have_fb && fb_f < f) { accept(fb_x, fb_f, fb_g, o, hist); if (status == RUNNING) status = CONVERGED; return; }
                status = CONVERGED;
                return;
            }
            thi = t;
            double tn = 0.5 * (tlo + thi);
            if (tlo == 0.0 && ok && lb_finite(ft)) {     // quadratic interpolation through f(0), f'(0), f(t)
                const double den = 2.0 * (ft - f - gd0 * t);
                if (den > 0.0) {
                    const double tq = -gd0 * t * t / den;
                    tn = fmin(fmax(tq, 0.1 * t), 0.5 * t);
                }
            }
            t = tn;
        }
        if (ls_trials >= o.max_ls || !(thi - tlo > 1e-16 * fmax(1.0, thi))) {
            if (have_fb && fb_f < f) { accept(fb_x, fb_f, fb_g, o, hist); return; }
            status = LS_STALL;
            return;
        }
        for (int i = 0; i < n; ++i) xt[i] = x[i] + t * d[i];
    }
};

}  // namespace gpcc
