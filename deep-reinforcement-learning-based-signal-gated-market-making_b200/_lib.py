"""ctypes binding of libsgmm_b200.so (include/sgmm.h).

There is no fallback: if the CUDA library is missing or fails to load, importing any compute
entry point raises ``SgmmLibraryError``.  Nothing here imports ``oracle/``.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libsgmm_b200.so")

OK, ERR_INVALID, ERR_CUDA, ERR_NOMEM, ERR_UNSUPPORTED = 0, -1, -2, -3, -4


class SgmmLibraryError(RuntimeError):
    pass


class SgmmError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"sgmm error {code}: {message}")
        self.code = code


f32p = C.POINTER(C.c_float)
f64p = C.POINTER(C.c_double)
i32p = C.POINTER(C.c_int32)
i64p = C.POINTER(C.c_int64)


class Population(C.Structure):
    _fields_ = [("hidden", C.c_int32), ("reserved", C.c_int32), ("count", C.c_int64),
                ("genomes", C.c_void_p), ("master", C.c_void_p),
                ("sigma", C.c_float), ("reserved2", C.c_float),
                ("seed", C.c_uint64), ("generation", C.c_uint64), ("first_index", C.c_int64)]


class RolloutParams(C.Structure):
    _fields_ = [("phi", C.c_double), ("fee_rate", C.c_double), ("precision", C.c_int32),
                ("flags", C.c_int32), ("units_per_lane", C.c_int32), ("warps_per_cta", C.c_int32)]


class Trace(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in
                ("off_a", "off_b", "adv_a", "adv_b", "fill_buy", "fill_sell", "inventory",
                 "cash", "reward", "pnl_reward", "inventory_reward", "fee_paid", "raw_a", "raw_b",
                 "spread", "wealth", "cum_reward", "skew", "cum_fees", "unrealized_pnl")]


class EnvState(C.Structure):
    _fields_ = [("phi", C.c_double), ("tick_size", C.c_double), ("fee_rate", C.c_double),
                ("inventory", C.c_int64), ("cash", C.c_double),
                ("i_max", C.c_int64), ("i_min", C.c_int64)]


class StepInfo(C.Structure):
    _fields_ = [("reward", C.c_double), ("pnl_reward", C.c_double),
                ("inventory_reward", C.c_double), ("fee_paid", C.c_double),
                ("fill_buy", C.c_int32), ("fill_sell", C.c_int32)]


class GaConfig(C.Structure):
    _fields_ = [("hidden", C.c_int32), ("use_arl", C.c_int32), ("pop_size", C.c_int64),
                ("shard_first", C.c_int64), ("shard_count", C.c_int64), ("shard_stride", C.c_int64),
                ("sigma", C.c_float), ("patience", C.c_int32),
                ("phi", C.c_double), ("fee_rate", C.c_double), ("seed", C.c_uint64),
                ("max_generations", C.c_int32), ("precision", C.c_int32)]


class GaStatus(C.Structure):
    _fields_ = [("generation", C.c_int32), ("stale", C.c_int32),
                ("sigma", C.c_float), ("adv_sigma", C.c_float),
                ("best_val", C.c_double), ("last_best_index", C.c_int64)]


class GaRun(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("phi", C.c_double), ("fee_rate", C.c_double),
                ("sigma", C.c_float), ("patience", C.c_int32)]


# every symbol include/sgmm.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "sgmm_version": (C.c_int, []),
    "sgmm_last_error": (C.c_char_p, []),
    "sgmm_abi_sizeof": (C.c_int, [C.c_int]),
    "sgmm_device_count": (C.c_int, []),
    "sgmm_device_info": (C.c_int, [C.c_int, i32p, i32p, i32p, C.POINTER(C.c_uint64)]),
    "sgmm_bundle_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double,
                                     C.c_int, C.c_void_p]),
    "sgmm_bundle_length": (C.c_int, [C.c_void_p, i64p]),
    "sgmm_bundle_device": (C.c_int, [C.c_void_p, i32p]),
    "sgmm_bundle_thresholds": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "sgmm_bundle_destroy": (C.c_int, [C.c_void_p]),
    "sgmm_rollout_population": (C.c_int, [C.c_void_p, C.POINTER(Population), C.POINTER(Population),
                                          C.POINTER(RolloutParams), C.c_void_p, C.c_void_p, C.c_void_p]),
    "sgmm_rollout_population_host": (C.c_int, [C.c_void_p, C.POINTER(Population), C.POINTER(Population),
                                               C.POINTER(RolloutParams), C.c_void_p, C.c_void_p, C.c_void_p]),
    "sgmm_rollout_population_host_async": (C.c_int, [C.c_void_p, C.POINTER(Population), C.POINTER(Population),
                                                     C.POINTER(RolloutParams), C.c_void_p, C.c_void_p, i32p]),
    "sgmm_rollout_wait": (C.c_int, [C.c_void_p, C.c_int32]),
    "sgmm_rollout_spec256_audit": (C.c_int, [C.c_void_p, C.POINTER(Population), C.POINTER(RolloutParams), C.c_void_p,
                                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "sgmm_rollout_tc_audit": (C.c_int, [C.c_void_p, C.POINTER(Population), C.POINTER(Population), C.POINTER(RolloutParams),
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "sgmm_rollout_trace": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                     C.POINTER(RolloutParams), C.POINTER(Trace), C.c_void_p, C.c_void_p,
                                     C.c_void_p]),
    "sgmm_rollout_trace_population": (C.c_int, [C.c_void_p, C.POINTER(Population), C.POINTER(Population), C.POINTER(RolloutParams),
                                                C.POINTER(Trace), C.c_void_p, C.c_void_p, C.c_void_p]),
    "sgmm_rollout_table": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(RolloutParams), C.POINTER(Trace), C.c_void_p,
                                     C.c_void_p, C.c_void_p]),
    "sgmm_env_init": (C.c_int, [C.POINTER(EnvState), C.c_double, C.c_double, C.c_double]),
    "sgmm_env_step_host": (C.c_int, [C.POINTER(EnvState), i64p, i64p, C.c_double, C.c_double, C.c_double,
                                     C.c_double, C.c_double, C.POINTER(StepInfo)]),
    "sgmm_env_step_host_real": (C.c_int, [C.POINTER(EnvState), f64p, i64p, C.c_double, C.c_double, C.c_double,
                                          C.c_double, C.c_double, C.POINTER(StepInfo)]),
    "sgmm_ga_create": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(GaConfig), C.c_void_p, C.c_void_p,
                                 C.c_int, C.c_void_p]),
    "sgmm_ga_destroy": (C.c_int, [C.c_void_p]),
    "sgmm_ga_buffers": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                  i64p, i32p, i32p]),
    "sgmm_ga_evaluate": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "sgmm_ga_select": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "sgmm_ga_generation": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "sgmm_ga_status_host": (C.c_int, [C.c_void_p, C.POINTER(GaStatus), C.c_void_p]),
    "sgmm_ga_master_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "sgmm_ga_history_host": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_void_p]),
    "sgmm_ga_create_sweep": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(GaConfig), C.c_int32, C.POINTER(GaRun), C.c_void_p,
                                       C.c_void_p, C.c_int, C.c_void_p]),
    "sgmm_ga_run_status_host": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(GaStatus), C.c_void_p]),
    "sgmm_ga_run_master_host": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "sgmm_ga_run_history_host": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_void_p, C.c_void_p]),
    "sgmm_bundle_windows": (C.c_int, [C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "sgmm_bundle_windows_host": (C.c_int, [C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                           C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_int, C.c_void_p]),
    "sgmm_trace_analytics": (C.c_int, [C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "sgmm_trace_analytics_host": (C.c_int, [C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_int, C.c_void_p]),
    "sgmm_measure_fp32_peak": (C.c_int, [C.c_int, f64p, C.c_void_p]),
}

_lib = None


def lib():
    """Load libsgmm_b200.so and type every entry point.  Fails loudly; never falls back."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise SgmmLibraryError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  There is no CPU fallback.")
        try:
            L = C.CDLL(LIB_PATH)
        except OSError as e:
            raise SgmmLibraryError(f"cannot load {LIB_PATH}: {e}") from e
        for name, (res, args) in SIGNATURES.items():
            try:
                fn = getattr(L, name)
            except AttributeError as e:
                raise SgmmLibraryError(f"{LIB_PATH} does not export {name}") from e
            fn.restype = res
            fn.argtypes = args
        for which, struct in enumerate((Population, RolloutParams, Trace, EnvState, StepInfo, GaConfig, GaStatus, GaRun)):
            if L.sgmm_abi_sizeof(which) != C.sizeof(struct):
                raise SgmmLibraryError(f"{LIB_PATH}: sizeof({struct.__name__}) is {L.sgmm_abi_sizeof(which)} in the library, "
                                       f"{C.sizeof(struct)} in the ctypes mirror -- rebuild the library (stale .so?)")
        _lib = L
    return _lib


_DEFERRED = []          # (destroy entry, handle) released while a CUDA graph was being captured


def _capturing() -> bool:
    try:
        import torch
        return torch.cuda.is_available() and torch.cuda.is_current_stream_capturing()
    except Exception:
        return False


def release(destroy: str, handle) -> None:
    """Destroy a bundle or GA handle (``destroy`` names its entry: sgmm_bundle_destroy, sgmm_ga_destroy).  The destroy entries
    free device memory and synchronise, which a stream capture in progress on this thread does not allow: the capture would
    be invalidated.  A handle released while the current stream captures a CUDA graph (typically an object the garbage
    collector finalises in the middle of ``torch.cuda.graph``) is therefore kept and destroyed at the next release outside
    a capture."""
    h = handle.value if isinstance(handle, C.c_void_p) else handle
    if h:
        _DEFERRED.append((destroy, h))
    if not _DEFERRED or _capturing():
        return
    L = lib()
    while _DEFERRED:
        name, p = _DEFERRED.pop()
        getattr(L, name)(C.c_void_p(p))


def check(code: int):
    if code != OK:
        msg = lib().sgmm_last_error()
        raise SgmmError(code, msg.decode() if msg else "")
    return code
