"""ctypes view of the C ABI in include/bmm_capi.h (libbmm_b200.so, built in-tree by build.py).

There is no CPU fallback: if the shared library is missing or there is no CUDA device the calls
raise.  Nothing here imports torch or the oracle.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BMM_LIB") or os.path.join(_HERE, "libbmm_b200.so")   # BMM_LIB: A/B builds of the same ABI

BMM_FP64, BMM_FP32 = 0, 1
FLAG_STABLE_SOFTMAX, FLAG_COMPACT_Z, FLAG_NO_Z_HISTORY, FLAG_GRID_PATH, FLAG_X_PACKED, FLAG_NO_TENSOR = 1, 2, 4, 8, 16, 32
FLAG_STEPHENS_FIXED = 64
SAMPLER_FULL, SAMPLER_STICKBREAKING, SAMPLER_COLLAPSED, SAMPLER_DP = 0, 1, 2, 3

ERRORS = {
    -1: "BMM_ERR_INVALID", -2: "BMM_ERR_CUDA", -3: "BMM_ERR_NOT_BINARY", -4: "BMM_ERR_BETA_GAMMA",
    -5: "BMM_ERR_NO_FREE_CLUSTER", -6: "BMM_ERR_DP_STATE", -7: "BMM_ERR_NCCL", -8: "BMM_ERR_UNSUPPORTED",
    -9: "BMM_ERR_PROB", -10: "BMM_ERR_TIMEOUT",
}

_dbl_p = C.POINTER(C.c_double)
_i32_p = C.POINTER(C.c_int32)


class Replay(C.Structure):
    _fields_ = [("u", _dbl_p), ("u_slots", C.c_int32), ("pi", _dbl_p), ("theta", _dbl_p), ("alpha", _dbl_p)]


class Args(C.Structure):
    _fields_ = [
        ("X", _i32_p), ("N", C.c_int32), ("P", C.c_int32), ("nsamples", C.c_int32), ("K", C.c_int32),
        ("alpha", C.c_double), ("beta", C.c_double), ("gamma", C.c_double), ("a", C.c_double), ("b", C.c_double),
        ("burnin", C.c_int32), ("relabel", C.c_int32), ("burnrelabel", C.c_int32), ("debug", C.c_int32),
        ("n_chains", C.c_int32), ("chain_offset", C.c_int32), ("seed", C.c_uint64), ("precision", C.c_int32),
        ("device", C.c_int32), ("flags", C.c_uint32), ("replay", C.POINTER(Replay)),
        ("n_global", C.c_int64), ("row_offset", C.c_int64), ("thin", C.c_int32), ("reserved_", C.c_int32),
    ]


class Init(C.Structure):
    _fields_ = [("pi", _dbl_p), ("theta", _dbl_p), ("z", _i32_p)]


class Out(C.Structure):
    _fields_ = [
        ("pi", _dbl_p), ("alpha", _dbl_p), ("permutations", _i32_p), ("z", _i32_p), ("theta", _dbl_p),
        ("z_original", _i32_p), ("theta_original", _dbl_p), ("probs", _dbl_p), ("loglik", _dbl_p),
        ("Q_final", _dbl_p), ("status", _i32_p), ("counts", _i32_p),
        ("z_freq", C.POINTER(C.c_uint32)), ("z_last", _i32_p),
    ]


EXPORTS = [
    "bmm_gibbs_full", "bmm_gibbs_stickbreaking", "bmm_gibbs_collapsed", "bmm_gibbs_dp", "bmm_stephens_batch",
    "bmm_stephens_online", "bmm_stephens_batch_ex", "bmm_stephens_online_ex", "bmm_assign", "bmm_assign_warp", "bmm_grid_cost", "bmm_rdirichlet", "bmm_predictive", "bmm_waic", "bmm_waic_kernel_ms", "bmm_loo", "bmm_loo_kernel_ms", "bmm_loglik_matrix", "bmm_debug_ws_trace", "bmm_debug_ws_cta", "bmm_debug_chain_kernel", "bmm_debug_chain_phases", "bmm_full_condprob", "bmm_plan_create", "bmm_plan_run",
    "bmm_plan_sync", "bmm_plan_elapsed_ms", "bmm_plan_fetch", "bmm_plan_destroy", "bmm_dist_unique_id",
    "bmm_dist_init", "bmm_dist_finalize", "bmm_dist_p2p_local", "bmm_dist_p2p_attach", "bmm_dist_p2p_detach", "bmm_plan_kernel_ms", "bmm_host_alloc", "bmm_host_free", "bmm_release_cache", "bmm_last_error", "bmm_device_count", "bmm_launch_count", "bmm_fetch_bytes", "bmm_version",
]

_lib = None


class BmmError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("%s (%d): %s" % (ERRORS.get(code, "BMM_ERR"), code, msg))
        self.code = code


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "%s is missing: build it with `python -m bmm_mcmc_b200.build` (nvcc, sm_100a). "
                "There is no CPU fallback." % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        L.bmm_last_error.restype = C.c_char_p
        L.bmm_version.restype = C.c_char_p
        L.bmm_launch_count.restype = C.c_uint64
        L.bmm_fetch_bytes.restype = C.c_uint64
        L.bmm_plan_create.argtypes = [C.c_int32, C.POINTER(Args), C.POINTER(Init), C.POINTER(C.c_void_p)]
        for f in ("bmm_plan_run", "bmm_plan_sync", "bmm_plan_destroy"):
            getattr(L, f).argtypes = [C.c_void_p]
        L.bmm_plan_fetch.argtypes = [C.c_void_p, C.POINTER(Out)]
        L.bmm_plan_elapsed_ms.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float)]
        L.bmm_plan_kernel_ms.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
        L.bmm_host_alloc.argtypes = [C.c_uint64, C.POINTER(C.c_void_p)]
        L.bmm_host_free.argtypes = [C.c_void_p]
        L.bmm_grid_cost.argtypes = [C.c_int64, C.c_int32, C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_int32, C.c_int32,
                                    C.POINTER(C.c_double)]
        L.bmm_waic.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _dbl_p, _dbl_p,
                               C.c_uint32, C.c_int32, _dbl_p, _dbl_p, _dbl_p, _dbl_p, _dbl_p]
        L.bmm_debug_chain_phases.argtypes = [C.POINTER(C.c_uint64), C.c_int64]
        L.bmm_waic_kernel_ms.argtypes = [C.POINTER(C.c_float), C.POINTER(C.c_int32)]
        L.bmm_loo.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _dbl_p, _dbl_p, _dbl_p,
                              C.c_uint32, C.c_int32, _dbl_p, _dbl_p, _dbl_p, _dbl_p]
        L.bmm_loo_kernel_ms.argtypes = [C.POINTER(C.c_float), C.POINTER(C.c_int32)]
        L.bmm_loglik_matrix.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _dbl_p, _dbl_p,
                                        C.c_uint32, C.c_int32, _dbl_p]
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise BmmError(rc, lib().bmm_last_error().decode())
