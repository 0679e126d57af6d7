"""ctypes binding of libials_b200.so (the C ABI declared in include/ials_b200.h).

There is no CPU fallback: if the CUDA library has not been built the import of
this module fails loudly, and creating a trainer without a GPU raises.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_float, c_int, c_int32, c_int64, c_ubyte, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libials_b200.so")

IALS_OK = 0
IALS_ERR_INVALID_ARGUMENT = 1
IALS_ERR_RUNTIME = 2
IALS_ERR_CUDA = 3
IALS_ERR_NOT_IMPLEMENTED = 4


class ModelConfigStruct(ctypes.Structure):
    """``ials_model_config`` (IALSLearningConfig.hpp:15-31)."""

    _fields_ = [
        ("K", c_int64), ("alpha0", c_float), ("reg", c_float), ("nu", c_float),
        ("init_stdev", c_float), ("random_seed", c_int32), ("loss_type", c_int32),
    ]


class SolverConfigStruct(ctypes.Structure):
    """``ials_solver_config`` (IALSLearningConfig.hpp:97-112)."""

    _fields_ = [
        ("n_threads", c_int64), ("solver_type", c_int32), ("reserved", c_int32),
        ("max_cg_steps", c_int64), ("ialspp_subspace_dimension", c_int64),
        ("ialspp_iteration", c_int64),
    ]


def _load() -> ctypes.CDLL:
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build the sm_100a CUDA library first "
            "(`python -m irspack_b200.build`).  irspack_b200 has no CPU fallback."
        )
    lib = ctypes.CDLL(LIB_PATH)
    H = c_void_p
    MC, SC = POINTER(ModelConfigStruct), POINTER(SolverConfigStruct)
    sigs = {
        "ials_last_error": (c_char_p, []),
        "ials_version": (c_char_p, []),
        "ials_device_count": (c_int, []),
        "ials_trainer_create": (c_int, [MC, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_int, POINTER(H)]),
        "ials_trainer_create_from_device_csr": (c_int, [MC, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_int, c_int, POINTER(H)]),
        "ials_trainer_create_from_factors": (c_int, [MC, c_int64, c_int64, c_void_p, c_void_p, c_int, POINTER(H)]),
        "ials_trainer_destroy": (None, [H]),
        "ials_trainer_set_stream": (c_int, [H, c_void_p]),
        "ials_trainer_step": (c_int, [H, SC]),
        "ials_trainer_step_async": (c_int, [H, SC]),
        "ials_trainer_sync": (c_int, [H]),
        "ials_trainer_step_io": (c_int, [H, SC, c_void_p, c_void_p, c_void_p, c_void_p]),
        "ials_trainer_half_step": (c_int, [H, c_int, SC]),
        "ials_trainer_gram": (c_int, [H, c_int, c_void_p]),
        "ials_trainer_user_scores": (c_int, [H, c_int64, c_int64, SC, c_void_p]),
        "ials_trainer_get_factors": (c_int, [H, c_int, c_void_p]),
        "ials_trainer_set_factors": (c_int, [H, c_int, c_void_p]),
        "ials_trainer_set_factor_rows": (c_int, [H, c_int, c_int64, c_int64, c_void_p, c_int]),
        "ials_trainer_set_user_rows_flagged": (c_int, [H, c_int64, c_int64, c_void_p]),
        "ials_trainer_get_factor_rows": (c_int, [H, c_int, c_int64, c_int64, c_void_p]),
        "ials_trainer_factors_device": (c_int, [H, c_int, POINTER(c_void_p), POINTER(c_int64), POINTER(c_int64), POINTER(c_int64)]),
        "ials_trainer_transform": (c_int, [H, c_int, c_int64, c_int64, c_void_p, c_void_p, c_void_p, SC, c_void_p]),
        "ials_trainer_compute_loss": (c_int, [H, SC, POINTER(c_float)]),
        "ials_trainer_set_features": (c_int, [H, c_int, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_int64]),
        "ials_trainer_feature_weight_rows": (c_int, [H, c_int, POINTER(c_int64)]),
        "ials_trainer_get_feature_weight": (c_int, [H, c_int, c_void_p]),
        "ials_trainer_set_feature_weight": (c_int, [H, c_int, c_int64, c_void_p]),
        "ials_trainer_transform_feature": (c_int, [H, c_int, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
        "ials_trainer_transform_with_feature": (c_int, [H, c_int, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, SC, c_void_p]),
        "ials_trainer_recommend": (c_int, [H, c_int64, c_int64, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
        "ials_trainer_recommend_allowed": (c_int, [H, c_int64, c_int64, c_int64, c_int, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
        "ials_trainer_recommend_users": (c_int, [H, c_void_p, c_int64, c_int64, c_int, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
        "ials_trainer_recommend_embeddings": (c_int, [H, c_void_p, c_int64, c_int64, c_int, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
        "ials_trainer_similar": (c_int, [H, c_int, c_void_p, c_int64, c_int64, c_int64, c_int, c_int, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
        "ials_trainer_rank_candidates": (c_int, [H, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
        "ials_trainer_candidate_scores": (c_int, [H, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p]),
        "ials_trainer_explain": (c_int, [H, c_int, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
        "ials_metrics_accumulate": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_int64, c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
        "ials_eval_set_create": (c_int, [H, c_int64, c_int64, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_int, POINTER(H)]),
        "ials_eval_set_destroy": (None, [H]),
        "ials_eval_set_reset": (c_int, [H, c_void_p]),
        "ials_eval_set_buffers": (c_int, [H, POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p), POINTER(c_int64), POINTER(c_int64)]),
        "ials_eval_set_diversity": (c_int, [H, c_void_p, c_void_p]),
        "ials_trainer_evaluate": (c_int, [H, H, c_int64, c_int64]),
        "ials_eval_set_create_cold": (c_int, [H, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_int, POINTER(H)]),
        "ials_trainer_evaluate_cold": (c_int, [H, H, SC, c_int64, c_int64]),
        "ials_topk_scores": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
        "ials_retrieve_recommend": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_int64, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
        "ials_weighted_gram": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_int64, c_int64, c_float, c_int, c_void_p, c_void_p]),
        "ials_weighted_gram256": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_int64, c_int64, c_float, c_int, c_void_p, c_void_p]),
        "ials_weighted_gram_jobs": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_float, c_int, c_void_p, c_void_p]),
        "ials_trainer_set_profiling": (c_int, [H, c_int]),
        "ials_trainer_get_timings": (c_int, [H, POINTER(ctypes.c_double), POINTER(c_int64)]),
        "ials_trainer_plan_stats": (c_int, [H, c_int, POINTER(c_int64)]),
        "ials_kernel_launch_count": (c_int64, []),
        "ials_trainer_create_sharded": (c_int, [MC, c_int64, c_int64, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, POINTER(H)]),
        "ials_trainer_shard_range": (c_int, [H, c_int, POINTER(c_int64), POINTER(c_int64)]),
        "ials_trainer_gram_partial": (c_int, [H, c_int, POINTER(c_void_p), POINTER(c_int64)]),
        "ials_trainer_solve_shard": (c_int, [H, c_int, SC]),
        "ials_trainer_set_shard_features": (c_int, [H, c_int, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_int64, POINTER(c_int)]),
        "ials_trainer_check_shard_step": (c_int, [H, SC, c_int, c_int]),
        "ials_trainer_feature_partials": (c_int, [H, c_int, POINTER(c_void_p), POINTER(c_int64), POINTER(c_void_p), POINTER(c_int64)]),
        "ials_trainer_feature_refit": (c_int, [H, c_int]),
        "ials_trainer_compute_loss_shard": (c_int, [H, SC, c_int, POINTER(ctypes.c_double)]),
        "ials_trainer_ipc_handle": (c_int, [H, c_int, POINTER(c_ubyte)]),
        "ials_trainer_ipc_open_peers": (c_int, [H, c_int, c_void_p, c_int, c_int]),
    }
    for name, (res, args) in sigs.items():
        fn = getattr(lib, name)  # AttributeError here == header / library mismatch
        fn.restype = res
        fn.argtypes = args
    return lib


lib = _load()


def check(status: int) -> None:
    """Map a C status to the exception the reference would raise
    (std::invalid_argument -> ValueError, std::runtime_error -> RuntimeError)."""
    if status == IALS_OK:
        return
    msg = (lib.ials_last_error() or b"").decode("utf-8", "replace")
    if status == IALS_ERR_INVALID_ARGUMENT:
        raise ValueError(msg)
    if status == IALS_ERR_NOT_IMPLEMENTED:
        raise NotImplementedError(msg)
    raise RuntimeError(msg)


def device_count() -> int:
    return int(lib.ials_device_count())


def version() -> str:
    return lib.ials_version().decode()
