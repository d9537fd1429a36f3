"""ctypes binding of libgpcc_b200.so (include/gpcc_b200.h).  No compute happens in Python; if the CUDA
library is missing or no B200 is visible every entry point raises -- there is no CPU fallback."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GPCC_B200_LIB") or os.path.join(_HERE, "libgpcc_b200.so")   # override: dev builds only

EXPORTS = [
    "gpcc_version", "gpcc_last_error", "gpcc_ctx_create", "gpcc_ctx_destroy", "gpcc_ctx_set_profiling",
    "gpcc_ctx_get_stats", "gpcc_ctx_device_count", "gpcc_problem_create", "gpcc_problem_destroy",
    "gpcc_problem_get_prior", "gpcc_loglik_batch", "gpcc_loglik_theta_batch", "gpcc_fit_batch",
    "gpcc_grid_posterior", "gpcc_getprobabilities", "gpcc_postb", "gpcc_predict", "gpcc_predict_loglik",
    "gpcc_fit_options_default", "gpcc_fit_state_create", "gpcc_fit_state_destroy", "gpcc_fit_state_postb",
    "gpcc_fit_state_predict", "gpcc_fit_state_predict_loglik", "gpcc_fit_state_factorisations",
    "gpcc_comm_unique_id", "gpcc_ctx_comm_init_rank", "gpcc_fit_state_sample", "gpcc_problem_set_method",
    "gpcc_ss_state_create", "gpcc_ss_state_destroy", "gpcc_ss_state_predict", "gpcc_ss_state_predict_loglik",
    "gpcc_ss_sample", "gpcc_ss_state_sample",
]


class FitOptions(C.Structure):
    _fields_ = [("max_iter", C.c_int), ("rhomin", C.c_double), ("rhomax", C.c_double),
                ("alpha_floor", C.c_double), ("gtol", C.c_double), ("ftol", C.c_double),
                ("history", C.c_int), ("transform_id", C.c_int), ("theta0_per_candidate", C.c_int),
                ("optimizer", C.c_int), ("nm_gtol", C.c_double)]


class Stats(C.Structure):
    _fields_ = [("ms_total", C.c_double), ("ms_eval_kernels", C.c_double), ("ms_assembly", C.c_double),
                ("ms_factor", C.c_double), ("ms_gradreduce", C.c_double), ("n_eval_launches", C.c_longlong),
                ("n_evals", C.c_longlong), ("n_evals_grad", C.c_longlong), ("path", C.c_int),
                ("n_devices", C.c_int), ("n_shared_prefix", C.c_longlong), ("n_tau_cache", C.c_longlong), ("assembly_bytes", C.c_longlong)]


class GpccError(RuntimeError):
    pass


_lib = None


def load():
    """Load the shared library (once).  Raises GpccError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise GpccError(f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(make -C gpcc_b200/csrc).  gpcc_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    dp, ip, vp = C.POINTER(C.c_double), C.POINTER(C.c_int), C.c_void_p
    lib.gpcc_version.restype = C.c_int
    lib.gpcc_last_error.restype = C.c_char_p
    lib.gpcc_ctx_create.argtypes = [C.c_int, ip, C.POINTER(vp)]
    lib.gpcc_ctx_destroy.argtypes = [vp]
    lib.gpcc_ctx_set_profiling.argtypes = [vp, C.c_int]
    lib.gpcc_ctx_get_stats.argtypes = [vp, C.POINTER(Stats)]
    lib.gpcc_ctx_device_count.argtypes = [vp]
    lib.gpcc_problem_create.argtypes = [vp, C.c_int, ip, dp, dp, dp, C.c_int, dp, dp, C.POINTER(vp)]
    lib.gpcc_problem_destroy.argtypes = [vp]
    lib.gpcc_problem_get_prior.argtypes = [vp, dp, dp]
    lib.gpcc_problem_set_method.argtypes = [vp, C.c_int]
    lib.gpcc_loglik_batch.argtypes = [vp, C.c_int, dp, dp, dp, C.c_int, dp, dp, ip]
    lib.gpcc_loglik_theta_batch.argtypes = [vp, C.c_int, dp, dp, C.POINTER(FitOptions), C.c_int, dp, dp, ip]
    lib.gpcc_fit_batch.argtypes = [vp, C.c_int, dp, C.c_int, dp, C.POINTER(FitOptions), dp, dp, dp, dp, ip, ip, ip]
    lib.gpcc_grid_posterior.argtypes = [vp, C.c_int, dp, dp, C.c_int, dp, C.POINTER(FitOptions), dp, dp, dp, dp, dp, ip, ip]
    lib.gpcc_getprobabilities.argtypes = [vp, C.c_int, dp, dp, dp]
    lib.gpcc_postb.argtypes = [vp, dp, dp, C.c_double, dp, dp]
    lib.gpcc_predict.argtypes = [vp, dp, dp, C.c_double, ip, dp, dp, dp, dp]
    lib.gpcc_predict_loglik.argtypes = [vp, dp, dp, C.c_double, ip, dp, dp, dp, dp, ip]
    lib.gpcc_fit_options_default.argtypes = [C.POINTER(FitOptions)]
    lib.gpcc_fit_state_create.argtypes = [vp, dp, dp, C.c_double, C.POINTER(vp)]
    lib.gpcc_fit_state_destroy.argtypes = [vp]
    lib.gpcc_fit_state_postb.argtypes = [vp, dp, dp]
    lib.gpcc_fit_state_predict.argtypes = [vp, ip, dp, dp, dp, dp]
    lib.gpcc_fit_state_predict_loglik.argtypes = [vp, ip, dp, dp, dp, dp, ip]
    lib.gpcc_fit_state_factorisations.argtypes = [vp]
    lib.gpcc_fit_state_sample.argtypes = [vp, C.c_ulonglong, C.c_int, dp, dp]
    lib.gpcc_ss_state_create.argtypes = [vp, dp, dp, C.c_double, C.POINTER(vp)]
    lib.gpcc_ss_state_destroy.argtypes = [vp]
    lib.gpcc_ss_state_predict.argtypes = [vp, ip, dp, dp, dp]
    lib.gpcc_ss_state_predict_loglik.argtypes = [vp, ip, dp, dp, dp, dp, ip]
    lib.gpcc_ss_sample.argtypes = [vp, dp, dp, C.c_double, C.c_ulonglong, C.c_int, dp, dp, dp]
    lib.gpcc_ss_state_sample.argtypes = [vp, ip, dp, C.c_ulonglong, C.c_int, dp, dp, dp]
    lib.gpcc_comm_unique_id.argtypes = [C.c_char_p]
    lib.gpcc_ctx_comm_init_rank.argtypes = [vp, C.c_int, C.c_int, C.c_char_p]
    for name in EXPORTS:
        if name not in ("gpcc_last_error", "gpcc_fit_state_factorisations"):
            getattr(lib, name).restype = C.c_int
    lib.gpcc_fit_state_factorisations.restype = C.c_longlong
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise GpccError(f"libgpcc_b200 error {rc}: {load().gpcc_last_error().decode(errors='replace')}")
