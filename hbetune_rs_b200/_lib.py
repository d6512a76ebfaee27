"""ctypes binding of libhbegp.so (include/hbegp.h).  There is no CPU fallback: a missing or
unloadable library is an ImportError, and every compute call fails on a box without a GPU."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("HBEGP_LIB") or os.path.join(_HERE, "libhbegp.so")  # HBEGP_LIB: A/B builds of the same library

F64, F32 = 0, 1
OK, NOT_PD = 0, 1
ERR_INVALID, ERR_CUDA, ERR_NOMEM, ERR_UNSUPPORTED, ERR_NO_CAPTURE = -1, -2, -3, -4, -5


class RunResult(C.Structure):
    _fields_ = [
        ("best_lml", C.c_double),
        ("best_eval", C.c_longlong),
        ("n_evals", C.c_longlong),
        ("final_f", C.c_double),
        ("status", C.c_int),
        ("reserved", C.c_int),
    ]


class AcqResult(C.Structure):
    _fields_ = [
        ("best_value", C.c_double),
        ("best_eval", C.c_longlong),
        ("n_evals", C.c_longlong),
        ("status", C.c_int),
        ("reserved", C.c_int),
    ]


class YNorm(C.Structure):
    _fields_ = [("amplitude", C.c_double), ("expected", C.c_double), ("projection", C.c_int), ("dtype", C.c_int)]


OBJECTIVE_FN = C.CFUNCTYPE(C.c_double, C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_void_p)
ALLREDUCE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(C.c_double), C.c_long)
BATCH_OBJECTIVE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double),
                                 C.POINTER(C.c_double), C.POINTER(C.c_int))

# name -> (restype, argtypes); must list every symbol include/hbegp.h declares
PROTOTYPES = {
    "hbegp_version": (C.c_char_p, []),
    "hbegp_last_error": (C.c_char_p, []),
    "hbegp_ctx_create": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]),
    "hbegp_ctx_destroy": (C.c_int, [C.c_void_p]),
    "hbegp_ctx_set_workspace_limit": (C.c_int, [C.c_void_p, C.c_ulonglong]),
    "hbegp_ctx_set_resident_models": (C.c_int, [C.c_void_p, C.c_int]),
    "hbegp_ctx_model_stats": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_longlong),
                                        C.POINTER(C.c_longlong)]),
    "hbegp_ctx_launch_count": (C.c_longlong, [C.c_void_p]),
    "hbegp_set_data": (C.c_int, [C.c_void_p, C.c_long, C.c_int, C.c_void_p, C.c_void_p]),
    "hbegp_set_data_device": (C.c_int, [C.c_void_p, C.c_long, C.c_int, C.c_void_p, C.c_void_p]),
    "hbegp_lml_grad_batch": (C.c_int, [C.c_void_p, C.c_double, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_void_p]),
    "hbegp_fit_runs": (C.c_int, [C.c_void_p, C.c_double, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                 C.POINTER(RunResult), C.c_void_p]),
    "hbegp_fit_runs_sharded": (C.c_int, [C.c_void_p, C.c_double, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                         C.c_int, C.c_int, ALLREDUCE_FN, C.c_void_p, C.POINTER(RunResult), C.c_void_p]),
    "hbegp_fit_runs_with": (C.c_int, [BATCH_OBJECTIVE_FN, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_int, C.c_int, C.c_int, ALLREDUCE_FN, C.c_void_p, C.POINTER(RunResult), C.c_void_p]),
    "hbegp_batcher_create": (C.c_int, [C.c_void_p, C.c_double, C.c_int, C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]),
    "hbegp_batcher_eval": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.POINTER(C.c_double), C.c_void_p, C.POINTER(C.c_int)]),
    "hbegp_batcher_leave": (C.c_int, [C.c_void_p, C.c_int, C.c_double]),
    "hbegp_batcher_results": (C.c_int, [C.c_void_p, C.POINTER(RunResult), C.c_void_p, C.POINTER(C.c_longlong)]),
    "hbegp_batcher_destroy": (C.c_int, [C.c_void_p]),
    "hbegp_comm_unique_id": (C.c_int, [C.c_void_p]),
    "hbegp_comm_init": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "hbegp_comm_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_double),
                                  C.POINTER(C.c_longlong)]),
    "hbegp_lml_grad_batch_sharded": (C.c_int, [C.c_void_p, C.c_double, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                               C.c_void_p, C.c_void_p, C.c_void_p]),
    "hbegp_predict_sharded": (C.c_int, [C.c_void_p, C.c_long, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_long)]),
    "hbegp_multi_create": (C.c_int, [C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]),
    "hbegp_multi_destroy": (C.c_int, [C.c_void_p]),
    "hbegp_multi_n_gpus": (C.c_int, [C.c_void_p]),
    "hbegp_multi_ctx": (C.c_void_p, [C.c_void_p, C.c_int]),
    "hbegp_multi_set_data": (C.c_int, [C.c_void_p, C.c_long, C.c_int, C.c_void_p, C.c_void_p]),
    "hbegp_multi_lml_grad_batch": (C.c_int, [C.c_void_p, C.c_double, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_void_p, C.c_void_p]),
    "hbegp_multi_fit_runs": (C.c_int, [C.c_void_p, C.c_double, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                       C.POINTER(RunResult), C.c_void_p]),
    "hbegp_multi_model_create": (C.c_int, [C.c_void_p, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.POINTER(C.c_void_p), C.POINTER(C.c_double), C.c_void_p, C.c_void_p]),
    "hbegp_multi_model_destroy": (C.c_int, [C.c_void_p]),
    "hbegp_multi_model_replica": (C.c_void_p, [C.c_void_p, C.c_int]),
    "hbegp_multi_predict": (C.c_int, [C.c_void_p, C.c_long, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_long)]),
    "hbegp_pick_best_run": (C.c_int, [C.c_int, C.POINTER(RunResult)]),
    "hbegp_model_create": (C.c_int, [C.c_void_p, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.POINTER(C.c_void_p), C.POINTER(C.c_double), C.c_void_p, C.c_void_p]),
    "hbegp_model_extend": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_double), C.c_void_p,
                                     C.c_void_p, C.POINTER(C.c_int)]),
    "hbegp_model_destroy": (C.c_int, [C.c_void_p]),
    "hbegp_model_n": (C.c_long, [C.c_void_p]),
    "hbegp_model_dim": (C.c_int, [C.c_void_p]),
    "hbegp_predict": (C.c_int, [C.c_void_p, C.c_long, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_long)]),
    "hbegp_predict_warn_values": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "hbegp_kernel_matrix": (C.c_int, [C.c_void_p, C.c_double, C.c_int, C.c_void_p, C.c_long, C.c_void_p, C.c_long, C.c_void_p,
                                      C.c_void_p]),
    "hbegp_kernel_theta_grad": (C.c_int, [C.c_void_p, C.c_double, C.c_int, C.c_void_p, C.c_long, C.c_void_p, C.c_void_p,
                                          C.c_void_p]),
    "hbegp_kernel_diag": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.c_long, C.c_void_p]),
    "hbegp_lbfgs_set_tolerances": (C.c_int, [C.c_double, C.c_double]),
    "hbegp_predict_device": (C.c_int, [C.c_void_p, C.c_long, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "hbegp_predict_mean_ei": (C.c_int, [C.c_void_p, C.POINTER(YNorm), C.c_long, C.c_void_p, C.c_double, C.c_void_p,
                                        C.c_void_p, C.POINTER(C.c_long), C.POINTER(C.c_long)]),
    "hbegp_predict_confidence_bound": (C.c_int, [C.c_void_p, C.POINTER(YNorm), C.c_long, C.c_void_p, C.c_double,
                                                 C.c_void_p, C.POINTER(C.c_long), C.POINTER(C.c_long)]),
    "hbegp_predict_grad": (C.c_int, [C.c_void_p, C.c_long, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.POINTER(C.c_long)]),
    "hbegp_predict_mean_ei_grad": (C.c_int, [C.c_void_p, C.POINTER(YNorm), C.c_long, C.c_void_p, C.c_double, C.c_void_p,
                                             C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_long)]),
    "hbegp_predict_confidence_bound_grad": (C.c_int, [C.c_void_p, C.POINTER(YNorm), C.c_long, C.c_void_p, C.c_double,
                                                      C.c_void_p, C.c_void_p, C.POINTER(C.c_long)]),
    "hbegp_acquire_ei": (C.c_int, [C.c_void_p, C.POINTER(YNorm), C.c_double, C.c_long, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_int, C.c_void_p, C.c_void_p, C.POINTER(AcqResult), C.POINTER(C.c_long),
                                   C.POINTER(C.c_longlong)]),
    "hbegp_acquire_confidence_bound": (C.c_int, [C.c_void_p, C.POINTER(YNorm), C.c_double, C.c_long, C.c_void_p, C.c_void_p,
                                                 C.c_void_p, C.c_int, C.c_void_p, C.POINTER(AcqResult), C.POINTER(C.c_long),
                                                 C.POINTER(C.c_longlong)]),
    "hbegp_minimize_by_gradient": (C.c_int, [OBJECTIVE_FN, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_int, C.POINTER(C.c_double)]),
    "hbegp_rng_seed": (None, [C.c_ulonglong, C.POINTER(C.c_ulonglong)]),
    "hbegp_rng_fork": (None, [C.POINTER(C.c_ulonglong), C.POINTER(C.c_ulonglong)]),
    "hbegp_rng_uniform": (C.c_double, [C.POINTER(C.c_ulonglong), C.c_double, C.c_double]),
    "hbegp_ynorm_fit": (C.c_int, [C.c_int, C.c_int, C.c_long, C.c_void_p, C.POINTER(C.c_double), C.c_void_p,
                                  C.POINTER(YNorm)]),
    "hbegp_ynorm_apply": (C.c_int, [C.POINTER(YNorm), C.c_int, C.c_long, C.c_void_p, C.c_void_p, C.c_void_p]),
    "hbegp_estimate_amplitude": (C.c_int, [C.c_int, C.c_long, C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "hbegp_expected_improvement": (C.c_double, [C.c_double, C.c_double, C.c_double]),
    "hbegp_expected_improvement_a": (C.c_int, [C.c_int, C.c_long, C.c_void_p, C.c_void_p, C.c_double, C.c_void_p]),
    "hbegp_normal_inverse_cdf": (C.c_double, [C.c_double, C.c_double, C.c_double]),
    "hbegp_bench_phase": (C.c_int, [C.c_void_p, C.c_double, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                    C.POINTER(C.c_float)]),
    "hbegp_debug_poison": (C.c_int, [C.c_void_p]),
    "hbegp_debug_factor": (C.c_int, [C.c_void_p, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.POINTER(C.c_int)]),
}


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C hbetune_rs_b200/csrc`).  hbetune_rs_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    return lib


lib = _load()


class HbegpError(RuntimeError):
    def __init__(self, code: int, where: str):
        msg = lib.hbegp_last_error().decode("utf-8", "replace")
        super().__init__(f"{where} failed with status {code}: {msg}")
        self.code = code


def check(code: int, where: str) -> int:
    if code < 0:
        raise HbegpError(code, where)
    return code


def allreduce_callback(fn):
    """Wraps ``fn(np.ndarray float64) -> None`` (in-place sum over all ranks) as an ``hbegp_allreduce_fn``."""
    import numpy as np

    def cb(_user, values, count):
        try:
            fn(np.ctypeslib.as_array(values, shape=(count,)))
            return 0
        except Exception as exc:  # noqa: BLE001 - must not unwind through C
            import sys
            print(f"hbegp all-reduce callback failed: {exc!r}", file=sys.stderr)
            return 1
    return ALLREDUCE_FN(cb)
