"""Loads bess_b200/libbess_b200.so (the C ABI declared in include/bess_b200.h) with ctypes.

There is no Python/CPU fallback: if the library is missing, or no CUDA device is visible when a compute entry point is
called, an exception is raised."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libbess_b200.so")
_lib = None

dp = C.POINTER(C.c_double)
ip = C.POINTER(C.c_int)


class BessB200Error(RuntimeError):
    pass


class Csc(C.Structure):
    """struct bess_b200_csc (include/bess_b200.h): a sparse design in compressed sparse column form"""
    _fields_ = [("colptr", C.c_void_p), ("rowidx", C.c_void_p), ("values", C.c_void_p), ("nnz", C.c_longlong)]


class Ext(C.Structure):
    """struct bess_b200_ext (include/bess_b200.h)"""
    _fields_ = [("fold_of_row", ip), ("cv_seed", C.c_uint), ("x_on_device", C.c_int), ("device", C.c_int),
                ("screening_A_out", ip), ("chosen_s_out", ip), ("stats_out", dp), ("profile", C.c_int),
                ("world", C.c_int), ("rank", C.c_int), ("col_lo", C.c_longlong), ("p_total", C.c_longlong),
                ("nccl_unique_id", C.c_void_p), ("chosen_lambda_out", dp), ("beta_out_zeroed", C.c_int), ("cv_reduce_over_ranks", C.c_int),
                ("cv_seed_set", C.c_int), ("tie_exact_out", ip), ("resident_out", dp), ("fold_shard", C.c_int),
                ("x_csc", C.POINTER(Csc)), ("sparse_sweeps_out", ip)]


_PYWRAP_ARGS = [dp, C.c_int, C.c_int, dp, C.c_int, C.c_int, dp, C.c_int, C.c_bool, C.c_int, C.c_int, C.c_int, C.c_int,
                C.c_int, C.c_bool, C.c_int, C.c_bool, C.c_int, ip, C.c_int, dp, C.c_int, ip, C.c_int, dp, C.c_int,
                C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, C.c_int, C.c_bool, C.c_int, C.c_int,
                ip, C.c_int, C.c_double]


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise BessB200Error(
            f"{SO_PATH} is missing: build it with `python -m bess_b200.build` (nvcc, sm_100a). "
            "bess_b200 has no CPU fallback.")
    lib = C.CDLL(SO_PATH)
    lib.bess_b200_last_error.restype = C.c_char_p
    lib.pywrap_bess.restype = None
    lib.pywrap_bess.argtypes = _PYWRAP_ARGS + [dp, C.c_int, dp, C.c_int, dp, C.c_int, dp, C.c_int, dp, dp, C.c_int,
                                               dp, C.c_int, dp, C.c_int, ip, C.c_int, ip]
    lib.bess_b200_fit.restype = C.c_int
    lib.bess_b200_fit.argtypes = _PYWRAP_ARGS + [dp, C.c_int, dp, dp, dp, C.POINTER(Ext)]
    lib.bess_b200_trace.restype = C.c_int
    lib.bess_b200_trace.argtypes = [ip, ip, dp, dp, dp, dp, C.c_int]
    lib.bess_b200_cv_fold_ids.argtypes = [C.c_int, C.c_int, C.c_uint, ip]
    lib.bessgpu_create.argtypes = [C.POINTER(C.c_void_p), C.c_int]
    lib.bessgpu_destroy.argtypes = [C.c_void_p]
    lib.bessgpu_load.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, dp, dp, C.c_int]
    lib.bessgpu_load_csc.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_longlong, C.c_int,
                                     dp, dp, C.c_int]
    lib.bessgpu_screen.argtypes = [C.c_void_p, C.c_int, ip, C.c_int, ip]
    lib.bessgpu_screen_local.argtypes = [C.c_void_p, C.c_int, ip, C.c_int, dp, ip, ip]
    lib.bessgpu_gather_columns.argtypes = [C.c_void_p, ip, ip, C.c_int, C.c_void_p, C.c_longlong]
    lib.bessgpu_normalize.argtypes = [C.c_void_p, C.c_int, C.c_int]
    lib.bessgpu_get_norm.argtypes = [C.c_void_p, dp, dp, dp]
    lib.bessgpu_design.argtypes = [C.c_void_p, dp]
    lib.bessgpu_set_groups.argtypes = [C.c_void_p, ip, C.c_int]
    lib.bessgpu_run_batch_groups.argtypes = [C.c_void_p, C.c_int, ip, C.c_int, C.c_int, C.c_double, ip, dp, ip, ip, dp,
                                             C.c_int]
    lib.bessgpu_setup_chains.argtypes = [C.c_void_p, C.c_int, ip, C.c_int, C.c_int, C.c_int, ip, C.c_int]
    lib.bessgpu_run_batch.argtypes = [C.c_void_p, C.c_int, ip, C.c_int, C.c_int, ip, dp, ip, dp]
    lib.bessgpu_losses.argtypes = [C.c_void_p, ip, ip, ip, C.c_int, dp]
    lib.bessgpu_time_dual_sweep.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_float), dp]
    lib.bessgpu_stats.argtypes = [C.c_void_p, dp]
    lib.bessgpu_sacrifice.argtypes = [C.c_void_p, ip, C.c_int, C.c_double, dp, ip]
    lib.bessgpu_topk.argtypes = [dp, C.c_int, C.c_int, ip, ip]
    lib.bessgpu_screen_select.argtypes = [dp, C.c_int, C.c_int, ip, ip]
    lib.bess_b200_shard_range.restype = None
    lib.bess_b200_shard_range.argtypes = [C.c_longlong, C.c_int, C.c_int, C.POINTER(C.c_longlong),
                                          C.POINTER(C.c_longlong)]
    lib.bess_b200_chain_owner.argtypes = [C.c_int, C.c_int]
    lib.bess_b200_fold_shard_chains.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, ip, ip]
    lib.bess_b200_fold_shard_chains.restype = C.c_int
    lib.bess_b200_nccl_unique_id.argtypes = [C.c_void_p]
    lib.bess_b200_trace_lambda.argtypes = [dp]
    lib.bess_b200_pgs_line_box.argtypes = [dp, dp, C.c_int, C.c_int, C.c_double, C.c_double, dp, dp]
    lib.bess_b200_gen_design.argtypes = [C.c_void_p, C.c_int, C.c_longlong, C.c_longlong, C.c_double, C.c_ulonglong, C.c_int]
    lib.bess_b200_gen_design_cortype.argtypes = [C.c_void_p, C.c_int, C.c_longlong, C.c_longlong, C.c_double, C.c_ulonglong, C.c_int,
                                                 C.c_int]
    lib.bess_b200_merge_candidates.argtypes = [dp, ip, C.c_int, C.c_int, ip]
    _lib = lib
    return lib


def last_error() -> str:
    return load().bess_b200_last_error().decode()


def check(rc: int):
    if rc != 0:
        raise BessB200Error(last_error())


def require_gpu():
    if load().bess_b200_device_count() < 1:
        raise BessB200Error("no CUDA device visible: bess_b200 computes on the GPU only (no CPU fallback)")
