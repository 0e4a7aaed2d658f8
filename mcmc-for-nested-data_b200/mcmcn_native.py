"""ctypes binding of libmcmcn.so (C ABI in include/mcmcn.h).

Thin by design (north star (5)): structs mirror the header one to one, every call
checks the return code and raises with mcmcn_last_error().  There is no CPU
fallback: if the library is missing or fails to load, importing callers get a
RuntimeError telling them to run ``python __graft_entry__.py``.

It also holds the host helpers that engine, posteriorSampling and sampleDiagnosis share: tensor
pointers for the ABI, the rank / world query, the contiguous chain-range rule and the host-thread count.
"""

import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MCMCN_LIB", os.path.join(HERE, "libmcmcn.so"))   # MCMCN_LIB: A/B builds of the same ABI

MAX_PARAMS = 17

OBJ_GAUSSIAN_DISTRIBUTION = 0
OBJ_LINEAR_REGRESSION = 1
OBJ_BERNOULLI_LOGIT = 2
OBJ_USER = 3

POOL_PARTIAL = 0
POOL_NONE = 1
POOL_COMPLETE = 2
POOLING_CODE = {"partial": POOL_PARTIAL, "none": POOL_NONE, "complete": POOL_COMPLETE}

PRIOR_NORM = 0
PRIOR_GAMMA = 1
PRIOR_UNIFORM = 2
PRIOR_EXPON = 3
PRIOR_HALFNORM = 4
PRIOR_LOGNORM = 5
PRIOR_CAUCHY = 6
PRIOR_T = 7
PRIOR_BETA = 8
PRIOR_INVGAMMA = 9
PRIOR_LAPLACE = 10
PRIOR_LOGISTIC = 11
PRIOR_CHI2 = 12

ERRORS = {-1: "invalid argument", -2: "CUDA error", -3: "unsupported", -4: "NVRTC error"}

c_void_p = ctypes.c_void_p


class Prior(ctypes.Structure):
    _fields_ = [("family", ctypes.c_int32), ("reserved", ctypes.c_int32),
                ("a", ctypes.c_double), ("loc", ctypes.c_double), ("scale", ctypes.c_double),
                ("log_scale", ctypes.c_double), ("c0", ctypes.c_double), ("b", ctypes.c_double)]


class Model(ctypes.Structure):
    _fields_ = [("objective", ctypes.c_int32), ("n_params", ctypes.c_int32),
                ("n_coef", ctypes.c_int32), ("precision", ctypes.c_int32),
                ("pooling", ctypes.c_int32), ("n_groups", ctypes.c_int32),
                ("n_tasks", ctypes.c_int32), ("n_obj_const", ctypes.c_int32),
                ("n_obs", ctypes.c_int64),
                ("data", c_void_p), ("group_off", c_void_p), ("group_nobs", c_void_p),
                ("task_group0", c_void_p), ("task_group0_host", c_void_p),
                ("group_off_host", c_void_p), ("obj_const", c_void_p),
                ("user_objective", c_void_p),
                ("tc_data", c_void_p), ("tc_group_off", c_void_p), ("tc_max_block_floats", ctypes.c_int64),
                ("prior", Prior * MAX_PARAMS),
                ("split", c_void_p), ("split_scratch", c_void_p)]


class State(ctypes.Structure):
    _fields_ = [("n_chains", ctypes.c_int32), ("stride", ctypes.c_int32),
                ("chain_id0", ctypes.c_int64),
                ("theta", c_void_p), ("scale", c_void_p), ("counts", c_void_p),
                ("ll", c_void_p), ("lprior", c_void_p), ("hyper", c_void_p)]


class RunArgs(ctypes.Structure):
    _fields_ = [("iter0", ctypes.c_int64), ("n_iter", ctypes.c_int32), ("burn", ctypes.c_int32),
                ("thin", ctypes.c_int32), ("tune_interval", ctypes.c_int32),
                ("seed", ctypes.c_uint64),
                ("tape_z", c_void_p), ("tape_u", c_void_p), ("tape_accept", c_void_p),
                ("tape_zmu", c_void_p), ("tape_qsig", c_void_p),
                ("trace_ll", c_void_p), ("trace_lp", c_void_p), ("trace_diff", c_void_p),
                ("trace_accept", c_void_p),
                ("store", c_void_p), ("store_dtype", ctypes.c_int32),
                ("use_lprior_override", ctypes.c_int32),
                ("store_row0", ctypes.c_int64), ("store_rows", ctypes.c_int64),
                ("timing", c_void_p), ("loglik_store", c_void_p)]


# name -> (restype, argtypes); every symbol include/mcmcn.h declares
PROTOTYPES = {
    "mcmcn_version": (ctypes.c_int, []),
    "mcmcn_last_error": (ctypes.c_char_p, []),
    "mcmcn_tile_capacity_bytes": (ctypes.c_int, []),
    "mcmcn_supported": (ctypes.c_int, [ctypes.c_int] * 4),
    "mcmcn_uses_tensor_core": (ctypes.c_int, [ctypes.POINTER(Model)]),
    "mcmcn_run": (ctypes.c_int, [ctypes.POINTER(Model), ctypes.POINTER(State),
                                 ctypes.POINTER(RunArgs), c_void_p]),
    "mcmcn_timing_collect": (ctypes.c_int, []),
    "mcmcn_group_loglik": (ctypes.c_int, [ctypes.POINTER(Model), ctypes.POINTER(State),
                                          c_void_p, c_void_p, c_void_p]),
    "mcmcn_pooled_nll": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, c_void_p, c_void_p, c_void_p]),
    "mcmcn_pointwise_loglik": (ctypes.c_int, [ctypes.POINTER(Model), ctypes.POINTER(State),
                                              c_void_p, c_void_p]),
    "mcmcn_diag_halfchains": (ctypes.c_int, [c_void_p, ctypes.c_int32, ctypes.c_int32, ctypes.c_int64, ctypes.c_int64,
                                             ctypes.c_int64, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32,
                                             c_void_p, c_void_p]),
    "mcmcn_diag_moments": (ctypes.c_int, [c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32,
                                          c_void_p, c_void_p, c_void_p]),
    "mcmcn_diag_variogram": (ctypes.c_int, [c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32,
                                            c_void_p, c_void_p]),
    "mcmcn_diag_rhat": (ctypes.c_int, [c_void_p, c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32,
                                       c_void_p, c_void_p]),
    "mcmcn_diag_ess": (ctypes.c_int, [c_void_p, c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32,
                                      c_void_p, c_void_p, c_void_p]),
    "mcmcn_diag_row_mean": (ctypes.c_int, [c_void_p, ctypes.c_int64, ctypes.c_int64, c_void_p, c_void_p]),
    "mcmcn_diag_sort_keys": (ctypes.c_int, [c_void_p, ctypes.c_int64, ctypes.c_int64, c_void_p]),
    "mcmcn_diag_median_hdi": (ctypes.c_int, [c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64,
                                             c_void_p, c_void_p]),
    "mcmcn_peak_fp32": (ctypes.c_int, [ctypes.POINTER(ctypes.c_double), c_void_p]),
    "mcmcn_peak_mufu": (ctypes.c_int, [ctypes.POINTER(ctypes.c_double), c_void_p]),
    "mcmcn_peak_tf32": (ctypes.c_int, [ctypes.POINTER(ctypes.c_double), c_void_p]),
    "mcmcn_user_objective_compile": (ctypes.c_int, [ctypes.c_char_p, ctypes.c_int32, ctypes.c_int32,
                                                    ctypes.c_int32, ctypes.c_int32,
                                                    ctypes.POINTER(c_void_p)]),
    "mcmcn_user_objective_free": (ctypes.c_int, [c_void_p]),
    "mcmcn_streams_create": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int64, ctypes.c_int32, ctypes.POINTER(c_void_p)]),
    "mcmcn_streams_free": (ctypes.c_int, [c_void_p]),
    "mcmcn_streams_uniform": (ctypes.c_int, [c_void_p, c_void_p, ctypes.c_int64, ctypes.c_int32, c_void_p, c_void_p,
                                             c_void_p, ctypes.c_int32]),
    "mcmcn_streams_normal": (ctypes.c_int, [c_void_p, c_void_p, ctypes.c_int64, c_void_p, c_void_p, ctypes.c_int32]),
    "mcmcn_streams_get_state": (ctypes.c_int, [c_void_p, ctypes.c_int64, c_void_p, ctypes.POINTER(ctypes.c_int32),
                                               ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_double)]),
    "mcmcn_streams_set_state": (ctypes.c_int, [c_void_p, ctypes.c_int64, c_void_p, ctypes.c_int32, ctypes.c_int32,
                                               ctypes.c_double]),
    "mcmcn_debug_philox": (ctypes.c_int, [c_void_p, c_void_p, c_void_p]),
    "mcmcn_debug_draws": (ctypes.c_int, [ctypes.c_int, ctypes.c_int64, ctypes.c_uint64, ctypes.c_double,
                                         c_void_p, c_void_p]),
}

DRAW_SWEEP_NORMALS, DRAW_SWEEP_UNIFORMS, DRAW_HYPER_NORMAL, DRAW_UNIT_INVGAMMA, DRAW_UNIFORM53 = range(5)

_lib = None


def load():
    """Load libmcmcn.so and attach the prototypes.  Raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "libmcmcn.so is not built (%s). Run `python __graft_entry__.py` at the repo root. "
            "There is no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        msg = load().mcmcn_last_error().decode("utf-8", "replace")
        raise RuntimeError("libmcmcn: %s (%s)" % (msg, ERRORS.get(rc, rc)))


def call(name, *args):
    check(getattr(load(), name)(*args))


# ---- host helpers shared by engine, posteriorSampling and sampleDiagnosis
def _ptr(t):
    """Device pointer of a tensor for the C ABI (None passes NULL)."""
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _rankWorld():
    """(rank, world size) under torch.distributed, (0, 1) without it."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def chainRange(n, rank, world):
    """Contiguous slice [lo, hi) of n items (chains; keys in the diagnostics' key-partitioned exchange) that a
    rank owns."""
    return (n * rank) // world, (n * (rank + 1)) // world


def _hostThreads(env):
    """Host copy threads of this process: an even share of the cores among the ranks of this box, 2..8."""
    share = (os.cpu_count() or 4) // max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))
    return int(os.environ.get(env, max(2, min(8, share // 2))))
