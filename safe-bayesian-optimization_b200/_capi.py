"""ctypes binding of libsbo_b200.so (the C ABI declared in include/sbo_b200.h).

There is no fallback: if the shared library is missing, or no B200 is visible,
importing works but creating a context raises.  The product path never touches
``oracle/``.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# SBO_B200_LIB: developer override to A/B-test another build of the same library (never a different backend)
LIB_PATH = os.environ.get("SBO_B200_LIB") or os.path.join(_HERE, "libsbo_b200.so")

MAX_D, MAX_G = 8, 8
UNSAFE_ALL, UNSAFE_ANY = 0, 1
MODE_LIPSCHITZ, MODE_FANTASY = 0, 1
PREC_FP64, PREC_TF32, PREC_TF32X3 = 0, 1, 2
# precision name -> (sbo_precision, keep_v of sbo_posterior) for the fantasy expander
PRECISIONS = {"fp64": (0, 1), "tf32": (1, 2), "tf32x3": (2, 3)}
ARGMAX_VAR0, ARGMIN_LCB0, ARGMIN_UCB0, ARGMIN_DIST = 0, 1, 2, 3
MASK_SAFE, MASK_MIN, MASK_UNSAFE, MASK_USER, MASK_EXPANDER, MASK_TARGET = 0, 1, 2, 3, 4, 5
# covariance function name (models/GP_Safe.GP kernel argument) -> enum sbo_kernel
KERNELS = {"RBF": 0, "Matern32": 1, "Matern52": 2}
BATCH_MAX_Q = 256                  # SBO_BATCH_MAX_Q: picks per batch acquisition
PHASES = ("model", "crosscov", "solve", "sets", "pairs", "argreduce", "pair_prep", "refine", "posterior_update")


class SetsResult(C.Structure):
    _fields_ = [("n_safe", C.c_int64), ("n_unsafe", C.c_int64), ("n_min", C.c_int64),
                ("min_ucb0", C.c_double), ("min_ucb0_idx", C.c_int64),
                ("min_lcb0", C.c_double), ("min_lcb0_idx", C.c_int64),
                ("minimizer_var", C.c_double), ("minimizer_idx", C.c_int64)]


class PairResult(C.Structure):
    _fields_ = [("best_idx", C.c_int64), ("best_value", C.c_double),
                ("per_idx", C.c_int64 * MAX_G), ("per_value", C.c_double * MAX_G),
                ("n_x", C.c_int64), ("n_z", C.c_int64),
                ("pairs_algorithmic", C.c_int64), ("pairs_evaluated", C.c_int64), ("n_hit", C.c_int64),
                ("n_ambiguous", C.c_int64), ("n_refined_safe", C.c_int64),
                ("n_undecided", C.c_int64), ("undecided_best_idx", C.c_int64), ("undecided_best_value", C.c_double)]


class StepResult(C.Structure):
    _fields_ = [("sets", SetsResult), ("L", C.c_double * MAX_G), ("pairs", PairResult),
                ("x_new_idx", C.c_int64), ("explore_idx", C.c_int64)]


class PairsInfo(C.Structure):
    _fields_ = [("n_x_local", C.c_int64), ("n_z_local", C.c_int64), ("row_doubles", C.c_int64), ("vrow_bytes", C.c_int64)]


class BatchPick(C.Structure):
    _fields_ = [("idx", C.c_int64), ("from_expander", C.c_int32), ("pad", C.c_int32),
                ("std_min", C.c_double), ("idx_min", C.c_int64), ("std_exp", C.c_double), ("idx_exp", C.c_int64)]


class UpdateInfo(C.Structure):
    _fields_ = [("rows", C.c_int64), ("recomputed", C.c_int32), ("pad", C.c_int32)]


class GooseBatchPick(C.Structure):
    _fields_ = [("idx", C.c_int64), ("explore", C.c_int32), ("pad", C.c_int32), ("safe_lcb", C.c_double), ("safe_idx", C.c_int64),
                ("target_lcb", C.c_double), ("target_idx", C.c_int64), ("dist", C.c_double)]


_P = C.c_void_p
_D = C.POINTER(C.c_double)
_I64 = C.POINTER(C.c_int64)
_U32 = C.POINTER(C.c_uint32)

# name -> (restype, argtypes); must list every function include/sbo_b200.h declares
SIGNATURES = {
    "sbo_create": (C.c_int, [C.c_int, C.POINTER(_P)]),
    "sbo_destroy": (C.c_int, [_P]),
    "sbo_last_error": (C.c_char_p, [_P]),
    "sbo_set_stream": (C.c_int, [_P, _P]),
    "sbo_version": (C.c_int, []),
    "sbo_set_model": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, _D, _D, _D, _D, _D, _D, _D]),
    "sbo_set_model_ex": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, _D, _D, _D, _D, _D, _D, _D]),
    "sbo_get_model": (C.c_int, [_P, _D, _D, _D]),
    "sbo_append_sample": (C.c_int, [_P, _D, _D]),
    "sbo_stable_minmax": (C.c_int, [_P, C.c_int, C.c_int, C.c_double, _I64, _D, _I64, _D]),
    "sbo_set_grid": (C.c_int, [_P, C.c_int, _I64, _D, _D]),
    "sbo_set_points": (C.c_int, [_P, C.c_int64, C.c_int, _D]),
    "sbo_set_shard": (C.c_int, [_P, C.c_int64, C.c_int64]),
    "sbo_point_coords": (C.c_int, [_P, C.c_int64, _D]),
    "sbo_posterior": (C.c_int, [_P, C.c_int, C.c_int, _D, _D]),
    "sbo_posterior_update": (C.c_int, [_P, _D, _D, C.POINTER(UpdateInfo)]),
    "sbo_point_posterior": (C.c_int, [_P, C.c_int64, _D, _D, _D]),
    "sbo_lipschitz": (C.c_int, [_P, _D]),
    "sbo_point_mean_grad": (C.c_int, [_P, C.c_int, C.c_int64, _D, _D]),
    "sbo_sets_pass1": (C.c_int, [_P, C.c_double, C.c_int, C.c_int, C.POINTER(SetsResult)]),
    "sbo_sets_pass2": (C.c_int, [_P, C.c_double, C.POINTER(SetsResult)]),
    "sbo_sets": (C.c_int, [_P, C.c_double, C.c_int, C.c_int, C.POINTER(SetsResult)]),
    "sbo_get_mask": (C.c_int, [_P, C.c_int, C.c_int, _U32]),
    "sbo_set_user_mask": (C.c_int, [_P, _U32]),
    "sbo_user_mask_ball": (C.c_int, [_P, C.c_int, _D, C.c_double]),
    "sbo_mask_dev": (C.c_int, [_P, C.c_int, C.c_int, C.POINTER(_P), _I64]),
    "sbo_posterior_dev": (C.c_int, [_P, C.POINTER(_P), C.POINTER(_P)]),
    "sbo_argreduce": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, _D, _I64, _D]),
    "sbo_expander": (C.c_int, [_P, C.c_int, C.c_int, C.c_double, _D, C.POINTER(PairResult), C.POINTER(C.c_int32)]),
    "sbo_goose_target": (C.c_int, [_P, C.c_double, _D, C.POINTER(PairResult)]),
    "sbo_goose_target_ex": (C.c_int, [_P, C.c_int, C.c_int, C.c_double, _D, C.POINTER(PairResult)]),
    "sbo_set_shard_cyclic": (C.c_int, [_P, C.c_int, C.c_int, C.c_int64, _I64]),
    "sbo_pairs_prepare": (C.c_int, [_P, C.c_int, C.c_int, C.c_double, _D, C.POINTER(PairsInfo)]),
    "sbo_pairs_export_dev": (C.c_int, [_P, _P, _P]),
    "sbo_pairs_import_dev": (C.c_int, [_P, C.c_int64, _P, _P]),
    "sbo_pairs_run_dev": (C.c_int, [_P, C.c_int, _P]),
    "sbo_pairs_set_segments": (C.c_int, [_P, C.c_int, C.c_int, _I64]),
    "sbo_mask_export_dev": (C.c_int, [_P, C.c_int, C.c_int, _P, C.c_int64]),
    "sbo_pairs_set_global_unsafe_dev": (C.c_int, [_P, _P, C.c_int64, C.c_int]),
    "sbo_pairs_finish_dev": (C.c_int, [_P, C.c_int, C.c_int64, _P, C.POINTER(PairResult), C.POINTER(C.c_int32)]),
    "sbo_comm_unique_id": (C.c_int, [_P]),
    "sbo_comm_init": (C.c_int, [_P, C.c_int, C.c_int, _P]),
    "sbo_comm_destroy": (C.c_int, [_P]),
    "sbo_safeopt_step_sharded": (C.c_int, [_P, C.c_double, C.c_int, C.c_int, C.c_int, _D, C.POINTER(StepResult)]),
    "sbo_goose_step_sharded": (C.c_int, [_P, C.c_double, C.c_int, _D, C.POINTER(StepResult)]),
    "sbo_goose_step_sharded_ex": (C.c_int, [_P, C.c_double, C.c_int, C.c_int, C.c_int, _D, C.POINTER(StepResult)]),
    "sbo_safeopt_batch": (C.c_int, [_P, C.c_int, C.POINTER(BatchPick), C.POINTER(C.c_int)]),
    "sbo_batch_prepare": (C.c_int, [_P, C.c_int, _I64]),
    "sbo_batch_local": (C.c_int, [_P, C.POINTER(BatchPick)]),
    "sbo_batch_commit": (C.c_int, [_P, C.c_int64]),
    "sbo_safeopt_batch_sharded": (C.c_int, [_P, C.c_int, C.POINTER(BatchPick), C.POINTER(C.c_int)]),
    "sbo_goose_batch": (C.c_int, [_P, C.c_int, C.POINTER(GooseBatchPick), C.POINTER(C.c_int)]),
    "sbo_goose_batch_prepare": (C.c_int, [_P, C.c_int, _I64]),
    "sbo_goose_batch_local": (C.c_int, [_P, C.POINTER(GooseBatchPick)]),
    "sbo_goose_batch_nearest": (C.c_int, [_P, C.c_int64, _I64, _D]),
    "sbo_goose_batch_commit": (C.c_int, [_P, C.c_int64, C.c_int64]),
    "sbo_goose_batch_sharded": (C.c_int, [_P, C.c_int, C.POINTER(GooseBatchPick), C.POINTER(C.c_int)]),
    "sbo_kernel_launches": (C.c_int64, [_P, C.c_int]),
    "sbo_mem_peak": (C.c_int64, [_P, C.c_int]),
    "sbo_phase_ms": (C.c_int, [_P, C.c_int, _D]),
    "sbo_refine_stats": (C.c_int, [_P, _I64, _I64]),
    "sbo_set_option": (C.c_int, [_P, C.c_char_p, C.c_int64]),
    "sbo_release": (C.c_int, [_P, C.c_int]),
    "sbo_nll_batch": (C.c_int, [_P, C.c_int, C.c_int, _D, _D, C.c_int, _D, _D]),
    "sbo_nll_batch_ex": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, _D, _D, C.c_int, _D, _D]),
}

_lib = None


def load():
    """Load libsbo_b200.so and attach the signatures.  Raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  There is no CPU fallback for this path.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)   # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def dptr(a):
    return a.ctypes.data_as(_D)
