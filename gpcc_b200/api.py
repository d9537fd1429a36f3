"""Python mirror of the reference interface for the hot path (see package docstring)."""
import ctypes as C
import math
import sys

import numpy as np

from . import _lib
from ._lib import FitOptions, GpccError, Stats, check

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)


def _d(a):
    return a.ctypes.data_as(_dp) if a is not None else None


def _i(a):
    return a.ctypes.data_as(_ip) if a is not None else None


def _f64(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None:
        a = a.reshape(shape)
    return a


# ---- the four kernels (src/util.jl:15-52): identity objects mapped to the C enum -------------------
class _Kernel:
    def __init__(self, name, kid):
        self.name, self.kid = name, kid

    def __repr__(self):
        return f"GPCC.{self.name}"


OU, rbf, matern32, matern52 = _Kernel("OU", 0), _Kernel("rbf", 1), _Kernel("matern32", 2), _Kernel("matern52", 3)
_KERNELS = {k.name: k for k in (OU, rbf, matern32, matern52)}


def _kernel_id(kernel):
    if isinstance(kernel, _Kernel):
        return kernel.kid
    if isinstance(kernel, str) and kernel in _KERNELS:
        return _KERNELS[kernel].kid
    raise GpccError(f"unsupported kernel {kernel!r}: expected one of GPCC.OU, GPCC.rbf, GPCC.matern32, "
                    "GPCC.matern52 (arbitrary kernel functions would need a CPU path, which does not exist)")


# ---- MiscUtil transforms used to build start points (gpccfixdelay_marginaliseb.jl:195-196) -----------
def _invmakepositive(y):
    y = np.asarray(y, dtype=np.float64)
    return y + np.log(-np.expm1(-y))


def _invtransformbetween(y, lo, hi):
    u = (np.asarray(y, dtype=np.float64) - lo) / (hi - lo)
    return np.log(u) - np.log1p(-u)


def initial_solutions(yarray, seed=1, numberofrestarts=1, initialrandom=5, rhomin=0.1, rhomax=20.0):
    """Start points theta0[restart][draw][L+1] drawn in the reference's order (:62, :166/:172, :188, :207).
    Julia's MersenneTwister stream is not reproducible here; numpy's default_rng(seed) is used instead, and
    the C ABI takes theta0 explicitly so a Julia caller passes its own draws."""
    rg = np.random.default_rng(seed)
    L = len(yarray)
    if numberofrestarts in (1, 2):
        rho0 = rg.uniform(rhomin + 1e-3, rhomax - 1e-3, numberofrestarts)
    else:
        rho0 = np.exp(np.linspace(np.log(rhomin + 1e-3), np.log(rhomax - 1e-3), numberofrestarts))
    var_y = np.array([np.var(np.asarray(a, dtype=np.float64), ddof=1) for a in yarray])
    out = np.empty((numberofrestarts, initialrandom, L + 1))
    for i in range(numberofrestarts):
        for j in range(initialrandom):
            alpha0 = var_y * (rg.random(L) * (1.2 - 0.8) + 0.8)
            out[i, j, :L] = _invmakepositive(alpha0)
            out[i, j, L] = _invtransformbetween(rho0[i], rhomin, rhomax)
    return out, rho0


class Context:
    """CUDA context(s) of the library: `ndev` devices, or explicit `devices` ids."""

    def __init__(self, ndev=1, devices=None, profiling=False):
        lib = _lib.load()
        self._h = C.c_void_p()
        ids = None
        if devices is not None:
            ids = np.ascontiguousarray(devices, dtype=np.int32)
            ndev = len(ids)
        check(lib.gpcc_ctx_create(int(ndev), _i(ids), C.byref(self._h)))
        if profiling:
            self.set_profiling(True)

    def set_profiling(self, on):
        check(_lib.load().gpcc_ctx_set_profiling(self._h, 1 if on else 0))

    def comm_init_rank(self, world, rank, unique_id):
        """Join a multi-process communicator (one process per GPU): see gpcc_ctx_comm_init_rank."""
        if len(unique_id) != 128:
            raise GpccError("the NCCL unique id is 128 bytes")
        check(_lib.load().gpcc_ctx_comm_init_rank(self._h, int(world), int(rank), bytes(unique_id)))
        self.world, self.rank = int(world), int(rank)

    @property
    def ndev(self):
        return _lib.load().gpcc_ctx_device_count(self._h)

    def stats(self):
        st = Stats()
        check(_lib.load().gpcc_ctx_get_stats(self._h, C.byref(st)))
        return {f: getattr(st, f) for f, _ in Stats._fields_}

    def getprobabilities(self, loglikel, logpriorpdfvalues=None):
        ll = _f64(loglikel)
        out = np.empty(ll.size)
        pr = None if logpriorpdfvalues is None else _f64(np.broadcast_to(logpriorpdfvalues, ll.shape))
        check(_lib.load().gpcc_getprobabilities(self._h, ll.size, _d(ll.ravel()), _d(pr.ravel()) if pr is not None else None, _d(out)))
        return out.reshape(ll.shape)

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            _lib.load().gpcc_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def comm_unique_id():
    """128-byte NCCL id drawn by rank 0; broadcast it to the other ranks with whatever the host program uses."""
    buf = C.create_string_buffer(128)
    check(_lib.load().gpcc_comm_unique_id(buf))
    return buf.raw


_default_ctx = None


def default_context():
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context(1)
    return _default_ctx


_OPTIMIZERS = {"lbfgs": 0, "neldermead": 1}


def _options(iterations, rhomin, rhomax, per_candidate=False, gtol=None, ftol=None, history=None, optimizer="lbfgs"):
    o = FitOptions()
    check(_lib.load().gpcc_fit_options_default(C.byref(o)))
    o.max_iter, o.rhomin, o.rhomax = int(iterations), float(rhomin), float(rhomax)
    o.theta0_per_candidate = 1 if per_candidate else 0
    if gtol is not None:
        o.gtol = gtol
    if ftol is not None:
        o.ftol = ftol
    if history is not None:
        o.history = history
    if optimizer not in _OPTIMIZERS:
        raise GpccError("optimizer must be 'lbfgs' (default) or 'neldermead' (the reference's, on the device)")
    o.optimizer = _OPTIMIZERS[optimizer]
    return o


_METHODS = {"dense": 0, "statespace": 1}


class Problem:
    """Device-resident data of one `gpcc` call (gpccfixdelay_marginaliseb.jl:85-98).

    `method` selects how the likelihood is evaluated: "dense" (default) factorises K + Sobs + B; "statespace" (OU,
    matern32, matern52) runs an exact Kalman filter in O(N) per evaluation (gpcc_problem_set_method), for light curves
    far beyond what a dense factorisation can hold.  `fit_state` and the prediction methods stay dense under either
    method; `statespace_fit_state` is the O(N) fit state of the state-space method and `statespace_sample` its O(N)
    draw."""

    def __init__(self, tarray, yarray, stdarray, kernel, ctx=None, method="dense"):
        self.ctx = ctx or default_context()
        self.L = len(tarray)
        if not (self.L == len(yarray) == len(stdarray)):
            raise GpccError("tarray, yarray, stdarray must have one inner array per band")   # :78
        self.n = np.array([len(a) for a in tarray], dtype=np.int32)
        for a, b in zip(yarray, stdarray):
            if len(a) != len(b):
                raise GpccError("band arrays differ in length")
        if any(len(a) != n for a, n in zip(yarray, self.n)):
            raise GpccError("band arrays differ in length")
        self.N = int(self.n.sum())
        t = _f64(np.concatenate([np.asarray(a, dtype=np.float64) for a in tarray]))
        y = _f64(np.concatenate([np.asarray(a, dtype=np.float64) for a in yarray]))
        s = _f64(np.concatenate([np.asarray(a, dtype=np.float64) for a in stdarray]))
        self.kernel_id = _kernel_id(kernel)
        self._h = C.c_void_p()
        check(_lib.load().gpcc_problem_create(self.ctx._h, self.L, _i(self.n), _d(t), _d(y), _d(s), self.kernel_id,
                                              None, None, C.byref(self._h)))
        self.mub, self.Sigmab = np.empty(self.L), np.empty(self.L)
        check(_lib.load().gpcc_problem_get_prior(self._h, _d(self.mub), _d(self.Sigmab)))
        self.method = "dense"
        if method != "dense":
            self.set_method(method)

    def set_method(self, method):
        """Switch between "dense" and "statespace" (see the class docstring)."""
        if method not in _METHODS:
            raise GpccError("method must be 'dense' or 'statespace'")
        check(_lib.load().gpcc_problem_set_method(self._h, _METHODS[method]))
        self.method = method

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            _lib.load().gpcc_problem_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- objective (:133-141) ---------------------------------------------------------------------
    def loglik_batch(self, delays, alpha, rho, want_grad=False):
        delays = _f64(delays, (-1, self.L))
        M = delays.shape[0]
        alpha = _f64(np.broadcast_to(_f64(alpha, (-1, self.L)), (M, self.L)))
        rho = _f64(np.broadcast_to(_f64(rho).reshape(-1), (M,)))
        ll = np.empty(M)
        grad = np.empty((M, self.L + 1)) if want_grad else None
        info = np.empty(M, dtype=np.int32)
        check(_lib.load().gpcc_loglik_batch(self._h, M, _d(delays), _d(alpha), _d(rho), 1 if want_grad else 0,
                                            _d(ll), _d(grad), _i(info)))
        return (ll, grad, info) if want_grad else (ll, info)

    def loglik_theta_batch(self, delays, theta, rhomin, rhomax, want_grad=False):
        delays = _f64(delays, (-1, self.L))
        M = delays.shape[0]
        theta = _f64(np.broadcast_to(_f64(theta, (-1, self.L + 1)), (M, self.L + 1)))
        o = _options(0, rhomin, rhomax)
        ll = np.empty(M)
        grad = np.empty((M, self.L + 1)) if want_grad else None
        info = np.empty(M, dtype=np.int32)
        check(_lib.load().gpcc_loglik_theta_batch(self._h, M, _d(delays), _d(theta), C.byref(o), 1 if want_grad else 0,
                                                  _d(ll), _d(grad), _i(info)))
        return (ll, grad, info) if want_grad else (ll, info)

    # ---- fit (:203-226) ------------------------------------------------------------------------------
    def fit_batch(self, delays, theta0, *, iterations, rhomin, rhomax, gtol=None, ftol=None, history=None, optimizer="lbfgs"):
        delays = _f64(delays, (-1, self.L))
        M = delays.shape[0]
        theta0 = _f64(theta0)
        per_cand = theta0.ndim == 3
        P = theta0.shape[-2]
        o = _options(iterations, rhomin, rhomax, per_cand, gtol, ftol, history, optimizer)
        res = dict(loglikel=np.empty(M), theta=np.empty((M, self.L + 1)), alpha=np.empty((M, self.L)), rho=np.empty(M),
                   iters=np.empty(M, dtype=np.int32), nfev=np.empty(M, dtype=np.int32), info=np.empty(M, dtype=np.int32))
        check(_lib.load().gpcc_fit_batch(self._h, M, _d(delays), P, _d(theta0), C.byref(o), _d(res["loglikel"]),
                                         _d(res["theta"]), _d(res["alpha"]), _d(res["rho"]), _i(res["iters"]),
                                         _i(res["nfev"]), _i(res["info"])))
        return res

    def grid_posterior(self, delays, theta0, *, iterations, rhomin, rhomax, logprior=None, gtol=None, ftol=None, optimizer="lbfgs"):
        delays = _f64(delays, (-1, self.L))
        M = delays.shape[0]
        theta0 = _f64(theta0)
        per_cand = theta0.ndim == 3
        P = theta0.shape[-2]
        o = _options(iterations, rhomin, rhomax, per_cand, gtol, ftol, None, optimizer)
        lp = None if logprior is None else _f64(logprior).reshape(M)
        res = dict(loglikel=np.empty(M), posterior=np.empty(M), theta=np.empty((M, self.L + 1)),
                   alpha=np.empty((M, self.L)), rho=np.empty(M), nfev=np.empty(M, dtype=np.int32),
                   info=np.empty(M, dtype=np.int32))
        check(_lib.load().gpcc_grid_posterior(self._h, M, _d(delays), _d(lp), P, _d(theta0), C.byref(o),
                                              _d(res["loglikel"]), _d(res["posterior"]), _d(res["theta"]),
                                              _d(res["alpha"]), _d(res["rho"]), _i(res["nfev"]), _i(res["info"])))
        return res

    # ---- postb (:248-252), predictTest (:259-343) -------------------------------------------------------
    def fit_state(self, delays, alpha, rho):
        """The state the reference's `pred` closures capture (:235-252): one factorisation, cached on the device."""
        return FitState(self, delays, alpha, rho)

    def statespace_fit_state(self, delays, alpha, rho):
        """O(N) fit state of the state-space method (gpcc_ss_state_*): per-point predictions and the test log-likelihood
        without a dense factorisation.  Needs method="statespace"."""
        return StateSpaceFitState(self, delays, alpha, rho)

    def statespace_sample(self, delays, alpha, rho, seed, nsamples=1, z=None, return_z=False):
        """Exact draws f ~ N(0, K + Sobs) in O(N) (gpcc_ss_sample), shape (nsamples, N) in input order.  Needs
        method="statespace".  z (nsamples, N, d+1), d = 1, 2, 3 for OU, matern32, matern52: the d process deviates and
        the noise deviate of every point, used instead of the generator (seed is then ignored).  return_z=True also
        returns the deviates used."""
        delays, alpha = _f64(delays, (self.L,)), _f64(alpha, (self.L,))
        d = {OU.kid: 1, matern32.kid: 2, matern52.kid: 3}.get(self.kernel_id, 1)
        ns = int(nsamples)
        if z is not None:
            z = _f64(z)
            if z.shape != (ns, self.N, d + 1):
                raise GpccError(f"z must have shape (nsamples, N, d+1) = {(ns, self.N, d + 1)}")
        f = np.empty((max(ns, 0), self.N))
        zo = np.empty((max(ns, 0), self.N, d + 1)) if return_z else None
        check(_lib.load().gpcc_ss_sample(self._h, _d(delays), _d(alpha), float(rho), int(seed) & (2 ** 64 - 1), ns, _d(z),
                                         _d(f), _d(zo)))
        return (f, zo) if return_z else f

    def postb(self, delays, alpha, rho):
        delays, alpha = _f64(delays, (self.L,)), _f64(alpha, (self.L,))
        mu, S = np.empty(self.L), np.empty((self.L, self.L))
        check(_lib.load().gpcc_postb(self._h, _d(delays), _d(alpha), float(rho), _d(mu), _d(S)))
        return mu, S

    def _pack_test(self, ttest_per_band):
        nt = np.array([len(a) for a in ttest_per_band], dtype=np.int32)
        if len(nt) != self.L:
            raise GpccError("ttest must have one inner array per band")
        tt = _f64(np.concatenate([np.asarray(a, dtype=np.float64) for a in ttest_per_band])) if nt.sum() else np.empty(0)
        return nt, tt

    def predict(self, delays, alpha, rho, ttest_per_band, full_cov=False):
        delays, alpha = _f64(delays, (self.L,)), _f64(alpha, (self.L,))
        nt, tt = self._pack_test(ttest_per_band)
        NT = int(nt.sum())
        mu, sd = np.empty(NT), np.empty(NT)
        S = np.empty((NT, NT)) if full_cov else None
        check(_lib.load().gpcc_predict(self._h, _d(delays), _d(alpha), float(rho), _i(nt), _d(tt), _d(mu), _d(sd), _d(S)))
        return mu, sd, S, nt

    def predict_loglik(self, delays, alpha, rho, ttest, ytest, stest):
        delays, alpha = _f64(delays, (self.L,)), _f64(alpha, (self.L,))
        nt, tt = self._pack_test(ttest)
        yt = _f64(np.concatenate([np.asarray(a, dtype=np.float64) for a in ytest]))
        st = _f64(np.concatenate([np.asarray(a, dtype=np.float64) for a in stest]))
        if not (len(tt) == len(yt) == len(st)):
            raise GpccError("test arrays differ in length")
        ll, info = C.c_double(), C.c_int()
        check(_lib.load().gpcc_predict_loglik(self._h, _d(delays), _d(alpha), float(rho), _i(nt), _d(tt), _d(yt), _d(st),
                                              C.byref(ll), C.byref(info)))
        return ll.value, info.value


class FitState:
    """Fitted state of one `gpcc` call on the device (gpcc_fit_state_*): the Cholesky factor of K + Sobs at (delays, alpha, rho),
    postb, and the scratch of the prediction calls.  The reference's closures capture KSobsB (:241) and re-factorise it on
    every call (:275, :283); here the N^3 work happens once, in the constructor."""

    def __init__(self, problem, delays, alpha, rho):
        self.problem = problem              # keeps the problem (and its context) alive
        self.L = problem.L
        self.delays, self.alpha, self.rho = _f64(delays, (self.L,)).copy(), _f64(alpha, (self.L,)).copy(), float(rho)
        self._h = C.c_void_p()
        check(_lib.load().gpcc_fit_state_create(problem._h, _d(self.delays), _d(self.alpha), self.rho, C.byref(self._h)))

    def postb(self):
        mu, S = np.empty(self.L), np.empty((self.L, self.L))
        check(_lib.load().gpcc_fit_state_postb(self._h, _d(mu), _d(S)))
        return mu, S

    def predict(self, ttest_per_band, full_cov=False):
        nt, tt = self.problem._pack_test(ttest_per_band)
        NT = int(nt.sum())
        mu, sd = np.empty(NT), np.empty(NT)
        S = np.empty((NT, NT)) if full_cov else None
        check(_lib.load().gpcc_fit_state_predict(self._h, _i(nt), _d(tt), _d(mu), _d(sd), _d(S)))
        return mu, sd, S, nt

    def predict_loglik(self, ttest, ytest, stest):
        nt, tt = self.problem._pack_test(ttest)
        yt = _f64(np.concatenate([np.asarray(a, dtype=np.float64) for a in ytest]))
        st = _f64(np.concatenate([np.asarray(a, dtype=np.float64) for a in stest]))
        if not (len(tt) == len(yt) == len(st)):
            raise GpccError("test arrays differ in length")
        ll, info = C.c_double(), C.c_int()
        check(_lib.load().gpcc_fit_state_predict_loglik(self._h, _i(nt), _d(tt), _d(yt), _d(st), C.byref(ll), C.byref(info)))
        return ll.value, info.value

    def sample(self, seed, nsamples=1, return_z=False):
        """Draws f ~ N(0, K + Sobs) at the state's hyper-parameters on the device: [nsamples][N] (simulatedata.jl:128-145)."""
        N = self.problem.N
        f = np.empty((int(nsamples), N))
        z = np.empty((int(nsamples), N)) if return_z else None
        check(_lib.load().gpcc_fit_state_sample(self._h, int(seed), int(nsamples), _d(f), _d(z)))
        return (f, z) if return_z else f

    @property
    def factorisations(self):
        return int(_lib.load().gpcc_fit_state_factorisations(self._h))

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            _lib.load().gpcc_fit_state_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class StateSpaceFitState:
    """Fit state of the state-space method on the device (gpcc_ss_state_*): the filtered moments and the backward-pass adjoint
    of the N merged training points at (delays, alpha, rho), O(N) memory.  Answers the per-point form of `pred` (means and
    standard deviations) and the test log-likelihood; the full predictive covariance needs the dense `fit_state`.  The
    state owns its data: it stays usable after its problem is closed.  `sample` draws the test values jointly from the
    predictive distribution, the route to any derived quantity without the full covariance."""

    def __init__(self, problem, delays, alpha, rho):
        self.problem = problem              # keeps the context alive
        self.L = problem.L
        self.delays, self.alpha, self.rho = _f64(delays, (self.L,)).copy(), _f64(alpha, (self.L,)).copy(), float(rho)
        self._h = C.c_void_p()
        check(_lib.load().gpcc_ss_state_create(problem._h, _d(self.delays), _d(self.alpha), self.rho, C.byref(self._h)))

    def predict(self, ttest_per_band, full_cov=False):
        if full_cov:
            raise GpccError("the state-space fit state gives per-point means and standard deviations only: the full "
                            "predictive covariance needs the dense fit_state")
        nt, tt = self.problem._pack_test(ttest_per_band)
        NT = int(nt.sum())
        mu, sd = np.empty(NT), np.empty(NT)
        check(_lib.load().gpcc_ss_state_predict(self._h, _i(nt), _d(tt), _d(mu), _d(sd)))
        return mu, sd, None, nt

    def predict_loglik(self, ttest, ytest, stest):
        nt, tt = self.problem._pack_test(ttest)
        yt = _f64(np.concatenate([np.asarray(a, dtype=np.float64) for a in ytest]))
        st = _f64(np.concatenate([np.asarray(a, dtype=np.float64) for a in stest]))
        if not (len(tt) == len(yt) == len(st)):
            raise GpccError("test arrays differ in length")
        ll, info = C.c_double(), C.c_int()
        check(_lib.load().gpcc_ss_state_predict_loglik(self._h, _i(nt), _d(tt), _d(yt), _d(st), C.byref(ll), C.byref(info)))
        return ll.value, info.value

    def sample(self, ttest_per_band, seed, nsamples=1, z=None, return_z=False):
        """Exact joint draws of the test values given the training data (gpcc_ss_state_sample), shape (nsamples, NT) with
        the bands concatenated as `predict` returns them: distributed as N(mu, Sigma) of the dense pred(::Vector{Vector})
        (:259-289), jitter included, in O(N + NT) per draw.  z (nsamples, (N+NT)(d+1) + L), d = 1, 2, 3 for OU, matern32,
        matern52: per sample, the d process deviates and the noise deviate of every training point (input order) and
        every test point (in the order of ttest_per_band), then the L shift deviates; used instead of the generator (seed
        is then ignored).  return_z=True also returns the deviates used, in the same shape."""
        nt, tt = self.problem._pack_test(ttest_per_band)
        NT, ns = int(nt.sum()), int(nsamples)
        d = {OU.kid: 1, matern32.kid: 2, matern52.kid: 3}.get(self.problem.kernel_id, 1)
        zp, K = (self.problem.N + NT) * (d + 1), (self.problem.N + NT) * (d + 1) + self.L
        zc = None
        if z is not None:
            z = _f64(z)
            if z.shape != (ns, K):
                raise GpccError(f"z must have shape (nsamples, (N+NT)(d+1) + L) = {(ns, K)}")
            zc = _f64(np.concatenate([z[:, :zp].ravel(), z[:, zp:].ravel()]))
        f = np.empty((max(ns, 0), NT))
        zo = np.empty(max(ns, 0) * K) if return_z else None
        check(_lib.load().gpcc_ss_state_sample(self._h, _i(nt), _d(tt), int(seed) & (2 ** 64 - 1), ns, _d(zc), _d(f),
                                               _d(zo)))
        if not return_z:
            return f
        zo = np.concatenate([zo[:ns * zp].reshape(ns, zp), zo[ns * zp:].reshape(ns, self.L)], axis=1)
        return f, zo

    def pred(self, ttest, ytest=None, stest=None):
        """The reference's `pred` forms (:259-343) except the full covariance (Vector{Vector} form, and the nearestposdef
        repair of a failed test likelihood), which raise GpccError."""
        return _pred_call(self, self.L, ttest, ytest, stest)

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            _lib.load().gpcc_ss_state_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MvNormal:
    """Stand-in for Distributions.MvNormal: what `postb` carries in the reference (:252)."""

    def __init__(self, mu, Sigma):
        self.mu, self.Sigma = np.asarray(mu), np.asarray(Sigma)

    mean = property(lambda self: self.mu)
    cov = property(lambda self: self.Sigma)

    def __repr__(self):
        return f"MvNormal(mu={self.mu}, Sigma={self.Sigma})"


class Uniform:
    """Stand-in for Distributions.Uniform (uniformpriordelay.jl:14)."""

    def __init__(self, a, b):
        self.a, self.b = float(a), float(b)

    def logpdf(self, x):
        x = np.asarray(x, dtype=np.float64)
        return np.where((x >= self.a) & (x <= self.b), -math.log(self.b - self.a), -np.inf)

    def __repr__(self):
        return f"Uniform(a={self.a}, b={self.b})"


def uniformpriordelay(*, L, z):
    """src/uniformpriordelay.jl:10-16 (scalar host arithmetic, stays on the host as in the reference)."""
    return Uniform(0.0, 10.0 ** 1.559 * (L * 10.0 ** (-44)) ** 0.549 * (1 + z))


def getprobabilities(loglikel, logpriorpdfvalues=None, ctx=None):
    """src/getprobabilities.jl:1-20, evaluated on the device; shape preserving."""
    return (ctx or default_context()).getprobabilities(loglikel, logpriorpdfvalues)


def _informuser(out, seed, iterations, numberofrestarts, initialrandom, rhomin, rhomax, Sigmab):
    # src/util.jl:1-11 -- the banner is observable behaviour (users @suppress it)
    out.write("Running with random seed %d\n" % seed)
    out.write("\t iterations             = %d\n" % iterations)
    out.write("\t initialrandom          = %d\n" % initialrandom)
    out.write("\t numberofrestarts       = %d\n" % numberofrestarts)
    out.write("\t JITTER                 = %e\n" % 1e-8)
    out.write("\t ρmin                   = %f\n" % rhomin)
    out.write("\t ρmax                   = %f\n" % rhomax)
    out.write("\t Σb                     = " + "".join("%.3f " % v for v in Sigmab) + "\n")


def _pred_call(state, L, ttest, ytest=None, stest=None):                                                # :259-343
    if ytest is not None:
        ll, info = state.predict_loglik(ttest, ytest, stest)
        if info != 0:
            # PosDefException branch of the reference (:323-341): nearestposdef(Sigma; minimumeigenvalue=1e-6), i.e.
            # eigenvalues clamped from below (src/UNUSED/gpcc.jl:294-300 spells it out), then logpdf.  The reference does
            # this repair in host code (MiscUtil) on an exceptional path; mu and Sigma still come from the device.
            mu_, _, S_, _ = state.predict(ttest, full_cov=True)
            S_ = S_ + np.diag(np.concatenate([_f64(a) for a in stest]) ** 2)
            return repaired_logpdf(mu_, S_, np.concatenate([_f64(a) for a in ytest]))
        return ll
    if len(ttest) > 0 and np.ndim(ttest[0]) > 0:                    # Vector{Vector}: (mu, Sigma) (:259-289)
        mu_, _, S_, _ = state.predict(ttest, full_cov=True)
        return mu_, S_
    tt = np.asarray(ttest, dtype=np.float64)                       # Vector: per band (mu, sigma) (:293-307)
    mu_, sd_, _, _ = state.predict([tt] * L)
    nt = len(tt)
    return [mu_[i * nt:(i + 1) * nt] for i in range(L)], [sd_[i * nt:(i + 1) * nt] for i in range(L)]


class _LazyPred:
    """`pred` of a state-space fit: the dense fit state (one N^3 factorisation) is only built on the first call or on the
    first access of `state`, so that a fit at large N that never predicts never factorises."""

    def __init__(self, problem, delays, alpha, rho, info):
        self._args, self._p, self._state, self.info = (delays, alpha, rho), problem, None, info

    @property
    def state(self):
        if self._state is None:
            self._state = self._p.fit_state(*self._args)
        return self._state

    def __call__(self, ttest, ytest=None, stest=None):
        return _pred_call(self.state, self._p.L, ttest, ytest, stest)


def gpcc(tarray, yarray, stdarray, *, kernel, delays, iterations, seed=1, numberofrestarts=1, initialrandom=5,
         rhomin=0.1, rhomax, theta0=None, ctx=None, verbose=True, problem=None, optimizer="lbfgs", method="dense"):
    """Drop-in for `gpcc` (gpccfixdelay_marginaliseb.jl:46-53): returns (loglikel, pred, (alpha, postb, rho)).
    method="statespace" fits with the Kalman filter (see Problem), takes postb from it, and builds the dense fit state
    behind `pred` only when `pred` is first used."""
    p = problem or Problem(tarray, yarray, stdarray, kernel, ctx, method)
    delays = _f64(delays)
    if delays.shape != (p.L,):
        raise GpccError("L == length(delays) violated")                                   # :78
    out = sys.stdout
    if verbose:
        _informuser(out, seed, iterations, numberofrestarts, initialrandom, rhomin, rhomax, p.Sigmab)   # :104
    if theta0 is None:
        theta0, rho0 = initial_solutions(yarray, seed, numberofrestarts, initialrandom, rhomin, rhomax)
        if verbose:
            out.write("\n\tInitial ρ values are:\n" + "".join("\t%f\n" % r for r in rho0))                # :179-181
    theta0 = _f64(theta0)
    if theta0.ndim == 2:
        theta0 = theta0[None]
    # restarts (:222-226): every restart is one more "candidate" with the same delays and its own start set
    R = theta0.shape[0]
    res = p.fit_batch(np.tile(delays, (R, 1)), theta0, iterations=iterations, rhomin=rhomin, rhomax=rhomax, optimizer=optimizer)
    best = int(np.argmax(res["loglikel"]))
    loglikel, alpha, rho = float(res["loglikel"][best]), res["alpha"][best].copy(), float(res["rho"][best])
    if verbose:
        out.write("\n\tOverall minimum is %f\n" % (-loglikel))                                          # :228
        out.write("(α, ρ) = unpack(paramopt) = (%s, %s)\n" % (alpha.tolist(), rho))                      # :235
    info = dict(nfev=int(res["nfev"][best]), iters=int(res["iters"][best]), status=int(res["info"][best]),
                theta=res["theta"][best].copy())
    if p.method == "statespace":
        mu, S = p.postb(delays, alpha, rho)                                                              # :248-252, by the filter
        return loglikel, _LazyPred(p, delays, alpha, rho, info), (alpha, MvNormal(mu, S), rho)
    state = p.fit_state(delays, alpha, rho)                      # K = delayedCovariance(...); KSobsB (:237-241), factorised once
    mu, S = state.postb()                                                                                # :248-252
    postb = MvNormal(mu, S)

    def pred(ttest, ytest=None, stest=None):                                                             # :259-343
        return _pred_call(state, p.L, ttest, ytest, stest)

    pred.state = state
    pred.info = info
    return loglikel, pred, (alpha, postb, rho)


def gpccgrid(tarray, yarray, stdarray, candidatedelays, *, kernel, iterations, seed=1, initialrandom=5, rhomin=0.1,
             rhomax, logprior=None, theta0=None, ctx=None, problem=None, method="dense"):
    """Additive batched entry replacing the README's `map`/`pmap` idiom (README.md:170-210, 285):
    candidatedelays is [M][L]; returns a dict with loglikel[M], posterior[M] (getprobabilities), alpha, rho."""
    p = problem or Problem(tarray, yarray, stdarray, kernel, ctx, method)
    if theta0 is None:
        theta0 = initial_solutions(yarray, seed, 1, initialrandom, rhomin, rhomax)[0][0]
    return p.grid_posterior(candidatedelays, theta0, iterations=iterations, rhomin=rhomin, rhomax=rhomax,
                            logprior=logprior)


def simulatedata_device(tarray, *, delays, alpha, b, rho=3.5, sigma=0.75, kernel=OU, seed=1, ctx=None, method="dense"):
    """The reference's simulator (src/simulatedata.jl:96-162) with the O(N^3) part on the device: the latent process is drawn
    from N(0, C + 1e-6 I), C = delayedCovariance(kernel, alpha, delays, rho, tarray) (:128; the 1e-6 stands in for the
    eigenvalue clamp of :132-138); scaling, offsets and observation noise (:151-159, alpha applied a second time as the
    reference does) are host arithmetic.  Returns (tarray, yarray, stdarray).
    method="dense" (default) draws through the tiled Cholesky and the generator of gpcc_fit_state_sample, for N in the
    thousands; method="statespace" draws exactly in O(N) through gpcc_ss_sample, for any N (OU, matern32, matern52)."""
    tarray = [_f64(a) for a in tarray]
    L = len(tarray)
    if method not in _METHODS:
        raise GpccError("method must be 'dense' or 'statespace'")
    dummy = [np.arange(len(a), dtype=np.float64) for a in tarray]              # the prior of b needs a variance; unused by the draw
    p = Problem(tarray, dummy, [np.full(len(a), 1e-3) for a in tarray], kernel, ctx, method)
    if method == "statespace":
        f = p.statespace_sample(delays, alpha, rho, seed)[0]
    else:
        st = p.fit_state(delays, alpha, rho)
        f = st.sample(seed, 1)[0]
        st.close()
    p.close()
    rg = np.random.default_rng(seed)
    y, mark = [], 0
    for l in range(L):
        n = len(tarray[l])
        y.append(f[mark:mark + n] * float(alpha[l]) + float(b[l]) + sigma * rg.standard_normal(n))
        mark += n
    return tarray, y, [sigma * np.ones(len(a)) for a in tarray]


def repaired_logpdf(mu, Sigma, y, minimumeigenvalue=1e-6):
    """logpdf(MvNormal(mu, nearestposdef(Sigma; minimumeigenvalue)), y): the PosDefException branch of the reference's test
    likelihood (gpccfixdelay_marginaliseb.jl:323-341; the eigenvalue clamp is spelled out in src/UNUSED/gpcc.jl:294-300)."""
    S = 0.5 * (np.asarray(Sigma, dtype=np.float64) + np.asarray(Sigma, dtype=np.float64).T)
    w, V = np.linalg.eigh(S)
    S = (V * np.maximum(w, minimumeigenvalue)) @ V.T
    c = np.linalg.cholesky(0.5 * (S + S.T))
    z = np.linalg.solve(c, np.asarray(y, dtype=np.float64) - np.asarray(mu, dtype=np.float64))
    return float(-0.5 * (len(z) * math.log(2.0 * math.pi) + 2.0 * np.sum(np.log(np.diag(c))) + z @ z))


def cv_folds(nper, numberoffolds=5, seedcv=1):
    """Fold assignment per band, each band partitioned on its own with seed seedcv + b (src/UNUSED/performcv.jl:66).  The
    reference takes its partitions from MiscUtil.CVindices (Julia RNG); a numpy permutation dealt round robin stands in
    for it here, and callers (the Julia shim) can pass their own `folds` instead."""
    folds = []
    for b, n in enumerate(nper):
        perm = np.random.default_rng(seedcv + b + 1).permutation(n)
        f = np.empty(n, dtype=np.int64)
        f[perm] = np.arange(n) % numberoffolds
        folds.append(f)
    return folds


def performcv(tobs, yobs, sobs, *, delays, kernel, iterations=1, seedcv=1, numberofrestarts=1, initialrandom=1,
              numberoffolds=5, rhomin=0.1, rhomax=20.0, folds=None, theta0=None, ctx=None, out=None, method="dense"):
    """K-fold cross-validation of the GPCC model at fixed delays, the retired consumer of `gpcc` + `pred(t, y, sigma)` in
    src/UNUSED/performcv.jl:41-139 (SURVEY.md 8f): per fold, fit on the training part and evaluate the test log-likelihood
    of the held-out part, both on the device.  Returns the vector of fold scores (to be fed to `getprobabilities`).
    `theta0[k]`: optional start set of fold k (restarts x draws x (L+1)), as in `gpcc`."""
    out = out or sys.stdout
    out.write("\nRunning CV with %d number of folds, random seed set to %d\n\n" % (numberoffolds, seedcv))       # :44
    if not (len(tobs) == len(yobs) == len(sobs)) or any(not (len(a) == len(b_) == len(c)) for a, b_, c in zip(tobs, yobs, sobs)):
        raise GpccError("tobs, yobs, sobs differ in shape")                                                       # :50-55
    if folds is None:
        folds = cv_folds([len(t) for t in tobs], numberoffolds, seedcv)
    fitness = np.zeros(numberoffolds)
    for k in range(numberoffolds):
        tr = [np.asarray(f) != k for f in folds]
        part = lambda arrs, masks: [_f64(a)[m] for a, m in zip(arrs, masks)]
        te = [~m for m in tr]
        out.write("\n--- fold %d train size is %d, test size is %d ---\n" % (k + 1, sum(int(m.sum()) for m in tr), sum(int(m.sum()) for m in te)))
        pred = gpcc(part(tobs, tr), part(yobs, tr), part(sobs, tr), kernel=kernel, delays=delays, iterations=iterations,
                    seed=seedcv, numberofrestarts=numberofrestarts, initialrandom=initialrandom, rhomin=rhomin, rhomax=rhomax,
                    theta0=None if theta0 is None else theta0[k], ctx=ctx, verbose=False, method=method)[1]                      # @suppress gpcc(...)[2] (:101)
        fitness[k] = pred(part(tobs, te), part(yobs, te), part(sobs, te))                                         # :104
        out.write("\t perf for fold %d is %f\n" % (k + 1, fitness[k]))
    return fitness
