"""ctypes binding of include/yelprec_b200.h (libyelprec_b200.so).

This is the whole Python<->CUDA boundary: plain pointers (tensor.data_ptr()), sizes and the current
CUDA stream handle. PyTorch only owns the device memory and the stream. There is NO CPU fallback:
if the library is missing the import of any compute entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

_LIB_NAME = "libyelprec_b200.so"
_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", _LIB_NAME)

# every symbol include/yelprec_b200.h declares (tests check the .so exports all of them)
SYMBOLS = (
    "yr_version", "yr_device_sm_count",
    "yr_mf_score", "yr_mf_score_bwd", "yr_bpr_loss_fwd", "yr_bpr_loss_bwd",
    "yr_bpr_mf_train_ws_bytes", "yr_bpr_mf_train", "yr_bpr_mf_validate",
    "yr_spmm_plan_size_h", "yr_spmm_plan_fill_h", "yr_spmm_plan_big_h", "yr_spmm_csr", "yr_ngcf_layer_fwd", "yr_ngcf_layer_bwd_ws_bytes", "yr_ngcf_layer_bwd",
    "yr_ngcf_dense_fwd", "yr_ngcf_dense_bwd",
    "yr_ngcf_tail", "yr_dense_opt_step", "yr_dense_opt_step_multi", "yr_ngcf_propagate", "yr_ngcf_train_step", "yr_ngcf_concat",
    "yr_ngcf_propagate_prefix", "yr_ngcf_train_step_ex",
    "yr_transpose_items", "yr_eval_ws_bytes", "yr_eval_topk_metrics", "yr_topk_masked_row", "yr_topk_masked_rows", "yr_topk_metrics", "yr_topk_merge",
    "yr_eval_tc_supported", "yr_eval_tc_ws_bytes", "yr_eval_topk_metrics_tc", "yr_eval_topk_metrics_tc_slice",
    "yr_cdae_ws_bytes", "yr_cdae_hidden", "yr_cdae_hidden_ex", "yr_cdae_output", "yr_cdae_step", "yr_cdae_step_ex", "yr_cdae_step_idx",
    "yr_nsbce_loss",
    "yr_shard_gather_rows", "yr_bpr_rows_grad", "yr_shard_accumulate", "yr_shard_step",
    "yr_shard_accumulate_sorted", "yr_adam_scalars", "yr_shard_step_sparse_adam", "yr_shard_gather_local", "yr_shard_catch_up",
    "yr_sample_negatives", "yr_laplacian_ws_bytes", "yr_laplacian_build",
    "yr_synth_user_rows", "yr_laplacian_binary_values",
    "yr_split_ws_bytes", "yr_split_sizes", "yr_split_per_user",
    "yr_recommend_ws_bytes", "yr_recommend_topk", "yr_recommend_subset_ws_bytes", "yr_recommend_subset_topk",
    "yr_recommend_topk_ex", "yr_recommend_subset_topk_ex", "yr_cdae_encode",
    "yr_recommend_geo_ws_bytes", "yr_recommend_geo_topk",
)

YR_OPT_SGD, YR_OPT_ADAM, YR_OPT_ADAMW = 0, 1, 2
YR_DTYPE_F32, YR_DTYPE_BF16 = 0, 1
# yr_dense_mode: where the NGCF d x d transforms run (per call / per trainer state)
YR_DENSE_FP32, YR_DENSE_TC_FWD, YR_DENSE_TC = 0, 1, 2
OPT_KINDS = {"sgd": YR_OPT_SGD, "adam": YR_OPT_ADAM, "adamw": YR_OPT_ADAMW}

_STATUS = {
    1000: "YR_ERR_BAD_ARG", 1001: "YR_ERR_BAD_DIM", 1002: "YR_ERR_BAD_OPT",
    1003: "YR_ERR_WORKSPACE", 1004: "YR_ERR_COOP",
}


class YrOpt(C.Structure):
    _fields_ = [("kind", C.c_int32), ("step", C.c_int32), ("lr", C.c_double), ("weight_decay", C.c_double),
                ("beta1", C.c_double), ("beta2", C.c_double), ("eps", C.c_double)]


class YrMfState(C.Structure):
    _fields_ = [("U", C.c_void_p), ("V", C.c_void_p),
                ("mU", C.c_void_p), ("vU", C.c_void_p), ("mV", C.c_void_p), ("vV", C.c_void_p),
                ("flagU", C.c_void_p), ("flagV", C.c_void_p),
                ("counters", C.c_void_p), ("err", C.c_void_p),
                ("ws", C.c_void_p), ("ws_bytes", C.c_size_t),
                ("nU", C.c_int64), ("nI", C.c_int64), ("d", C.c_int32), ("deterministic", C.c_int32)]


YR_SPMM_CHUNK = 128


class YrCsr(C.Structure):
    _fields_ = [("n_rows", C.c_int64), ("nnz", C.c_int64),
                ("rowptr", C.c_void_p), ("col", C.c_void_p), ("val", C.c_void_p),
                ("n_chunks", C.c_int32),
                ("chunk_desc", C.c_void_p),
                ("n_split_rows", C.c_int32),
                ("split_row", C.c_void_p), ("split_ptr", C.c_void_p), ("partials", C.c_void_p),
                ("split_count", C.c_void_p),
                ("n_big_rows", C.c_int32), ("big_split_idx", C.c_void_p), ("reserve_sms", C.c_int32)]


class YrShardState(C.Structure):
    _fields_ = [("T", C.c_void_p), ("m", C.c_void_p), ("v", C.c_void_p), ("gscratch", C.c_void_p),
                ("flags", C.c_void_p), ("rows_list", C.c_void_p), ("counters", C.c_void_p),
                ("row0", C.c_int64), ("row1", C.c_int64), ("d", C.c_int32)]


class YrCdaeTensors(C.Structure):
    _fields_ = [("Wh", C.c_void_p), ("bh", C.c_void_p), ("Vu", C.c_void_p), ("Wo", C.c_void_p), ("bo", C.c_void_p)]


YR_NGCF_MAX_LAYERS = 7
_PL = C.c_void_p * YR_NGCF_MAX_LAYERS
_PL1 = C.c_void_p * (YR_NGCF_MAX_LAYERS + 1)


class YrNgcfState(C.Structure):
    _fields_ = [("nU", C.c_int64), ("nI", C.c_int64), ("d", C.c_int32), ("n_layers", C.c_int32),
                ("L", YrCsr), ("LT", YrCsr),
                ("E", _PL1), ("LE", _PL), ("G", _PL1), ("T", C.c_void_p),
                ("W1", _PL), ("W2", _PL), ("dW1", _PL), ("dW2", _PL),
                ("mE", C.c_void_p), ("vE", C.c_void_p),
                ("mW1", _PL), ("vW1", _PL), ("mW2", _PL), ("vW2", _PL),
                ("E_dev", C.c_void_p), ("G_dev", C.c_void_p),
                ("ws", C.c_void_p), ("ws_bytes", C.c_size_t),
                ("loss", C.c_void_p), ("err", C.c_void_p),
                ("row_flag", C.c_void_p), ("row_list", C.c_void_p), ("row_count", C.c_void_p), ("row_list_cap", C.c_int64),
                ("dense_mode", C.c_int32), ("top_rows_mode", C.c_int32)]


class YelprecError(RuntimeError):
    pass


_lib: Optional[C.CDLL] = None


def lib_path() -> str:
    return _LIB_PATH


def load() -> C.CDLL:
    """Load the shared library (once). Raises if it was not built — never falls back to anything."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise YelprecError(
            f"{_LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C yelprecommendation_b200/csrc`. There is no CPU fallback.")
    lib = C.CDLL(_LIB_PATH)
    p, i32, i64, f32, sz = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_size_t
    sig = {
        "yr_version": (C.c_int, []),
        "yr_device_sm_count": (C.c_int, [C.POINTER(C.c_int)]),
        "yr_mf_score": (C.c_int, [p, p, i64, i64, i32, p, p, i64, p, p, p]),
        "yr_mf_score_bwd": (C.c_int, [p, p, i64, i64, i32, p, p, i64, p, p, p, p]),
        "yr_bpr_loss_fwd": (C.c_int, [p, p, i64, p, p]),
        "yr_bpr_loss_bwd": (C.c_int, [p, p, i64, p, p, p, p]),
        "yr_bpr_mf_train_ws_bytes": (sz, [i64, i32, i32]),
        "yr_bpr_mf_train": (C.c_int, [C.POINTER(YrMfState), C.POINTER(YrOpt), p, p, p, i64, i32, p, p, p]),
        "yr_bpr_mf_validate": (C.c_int, [p, p, i64, i64, i32, p, p, p, i64, i32, p, p, p, p]),
        "yr_spmm_plan_size_h": (C.c_int, [p, i64, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)]),
        "yr_spmm_plan_fill_h": (C.c_int, [p, i64, p, p, p]),
        "yr_spmm_plan_big_h": (C.c_int, [p, i64, C.POINTER(i32), p]),
        "yr_spmm_csr": (C.c_int, [C.POINTER(YrCsr), i32, p, p, i32, p]),
        "yr_ngcf_layer_fwd": (C.c_int, [C.POINTER(YrCsr), i32, p, p, p, f32, p, p, i32, p]),
        "yr_ngcf_layer_bwd_ws_bytes": (sz, [i32]),
        "yr_ngcf_layer_bwd": (C.c_int, [C.POINTER(YrCsr), i32, p, p, p, p, p, p, f32, p, p, p, p, p, sz, i32, p]),
        "yr_ngcf_dense_fwd": (C.c_int, [i32, i64, p, p, p, p, f32, p, i32, p]),
        "yr_ngcf_dense_bwd": (C.c_int, [i32, i64, p, p, p, p, p, p, f32, p, p, p, p, p, sz, i32, p]),
        "yr_ngcf_tail": (C.c_int, [p, p, i32, i64, i64, i32, p, p, p, i64, p, p, p, p, p, p]),
        "yr_dense_opt_step": (C.c_int, [p, p, p, p, i64, C.POINTER(YrOpt), p]),
        "yr_dense_opt_step_multi": (C.c_int, [i32, p, p, p, p, p, C.POINTER(YrOpt), i32, p]),
        "yr_ngcf_propagate": (C.c_int, [C.POINTER(YrNgcfState), f32, p]),
        "yr_ngcf_train_step": (C.c_int, [C.POINTER(YrNgcfState), C.POINTER(YrOpt), f32, p, p, p, i64, p, p]),
        "yr_ngcf_propagate_prefix": (C.c_int, [C.POINTER(YrNgcfState), f32, i32, p]),
        "yr_ngcf_train_step_ex": (C.c_int, [C.POINTER(YrNgcfState), C.POINTER(YrOpt), f32, p, p, p, i64, p, i32, p]),
        "yr_ngcf_concat": (C.c_int, [p, i32, i64, i32, p, p]),
        "yr_topk_masked_row": (C.c_int, [p, i64, p, i64, i32, p, p]),
        "yr_topk_masked_rows": (C.c_int, [p, i64, i64, i64, p, p, f32, i32, p, p, sz, p]),
        "yr_topk_metrics": (C.c_int, [p, i64, i64, p, p, p, p, i32, p, p, p]),
        "yr_topk_merge": (C.c_int, [p, p, i32, i64, i32, p, p, p, p]),
        "yr_transpose_items": (C.c_int, [p, i64, i32, p, i64, p]),
        "yr_eval_ws_bytes": (sz, [i64, i32, i32]),
        "yr_eval_topk_metrics": (C.c_int, [p, i64, p, i64, i64, i32, p, i64, p, p, p, p, p, p, i32,
                                           p, p, p, p, p, sz, p, p]),
        "yr_cdae_ws_bytes": (sz, [i64, i64]),
        "yr_cdae_hidden": (C.c_int, [C.POINTER(YrCdaeTensors), i64, i64, i32, p, p, p, i64, p, i64, p, sz, p, p]),
        "yr_cdae_hidden_ex": (C.c_int, [C.POINTER(YrCdaeTensors), i64, i64, i32, i32, p, p, p, i64, p, i64, p, sz, p, p]),
        "yr_cdae_output": (C.c_int, [C.POINTER(YrCdaeTensors), i64, i32, p, i64, i64, p, p]),
        "yr_cdae_step": (C.c_int, [C.POINTER(YrCdaeTensors), C.POINTER(YrCdaeTensors), C.POINTER(YrCdaeTensors),
                                   C.POINTER(YrCdaeTensors), C.POINTER(YrOpt), i64, i64, i32, p, p, p, p, p, i64, p, p,
                                   p, sz, p, p]),
        "yr_cdae_step_ex": (C.c_int, [C.POINTER(YrCdaeTensors), C.POINTER(YrCdaeTensors), C.POINTER(YrCdaeTensors),
                                      C.POINTER(YrCdaeTensors), C.POINTER(YrOpt), i64, i64, i32, i32, p, p, p, p, p, i64, p,
                                      p, p, sz, p, p]),
        "yr_cdae_step_idx": (C.c_int, [C.POINTER(YrCdaeTensors), C.POINTER(YrCdaeTensors), C.POINTER(YrCdaeTensors),
                                       C.POINTER(YrCdaeTensors), C.POINTER(YrOpt), i64, i64, i32, i32, p, p, p, p, p, p, p, i64,
                                       p, p, p, sz, p, p]),
        "yr_nsbce_loss": (C.c_int, [p, p, p, i64, p, p, sz, p]),
        "yr_laplacian_ws_bytes": (sz, [i64, i64, i64]),
        "yr_laplacian_build": (C.c_int, [p, p, p, i64, i64, i64, p, p, p, p, sz, p, p]),
        "yr_synth_user_rows": (C.c_int, [C.c_uint64, i64, i64, C.c_double, C.c_double, C.c_double, i32, i32, p, p, p, p]),
        "yr_laplacian_binary_values": (C.c_int, [p, i64, p, p, p, p, p]),
        "yr_split_ws_bytes": (sz, [i32]),
        "yr_split_sizes": (C.c_int, [p, i64, p, p, p, p]),
        "yr_split_per_user": (C.c_int, [p, p, i64, i32, C.c_uint32, p, p, p, p, p, p, p, sz, p, p]),
        "yr_sample_negatives": (C.c_int, [p, i64, p, p, i64, i64, C.c_uint64, C.c_uint64, i32, p, p, p]),
        "yr_shard_gather_rows": (C.c_int, [p, i64, i64, i64, i32, p, i64, p, i64, p, p]),
        "yr_bpr_rows_grad": (C.c_int, [p, i32, i64, i64, i64, p, p, p]),
        "yr_shard_accumulate": (C.c_int, [C.POINTER(YrShardState), C.POINTER(YrOpt), p, i64, p, i64, p]),
        "yr_shard_step": (C.c_int, [C.POINTER(YrShardState), C.POINTER(YrOpt), i64, p]),
        "yr_shard_accumulate_sorted": (C.c_int, [C.POINTER(YrShardState), C.POINTER(YrOpt), p, p, i64, p, i64, i32, p]),
        "yr_shard_catch_up": (C.c_int, [C.POINTER(YrShardState), C.POINTER(YrOpt), p, i32, p, p, i64, p]),
        "yr_shard_gather_local": (C.c_int, [p, p, i32, p, p, i64, p, i64, p]),
        "yr_adam_scalars": (C.c_int, [C.POINTER(YrOpt), i32, p, p]),
        "yr_shard_step_sparse_adam": (C.c_int, [C.POINTER(YrShardState), C.POINTER(YrOpt), p, i32, p, i64, i32, p]),
        "yr_eval_tc_supported": (C.c_int, [i32, i32]),
        "yr_eval_tc_ws_bytes": (sz, [i64]),
        "yr_eval_topk_metrics_tc": (C.c_int, [p, i64, p, p, i64, i64, i32, p, i64, p, p, p, p, p, p, i32,
                                              p, p, p, p, p, sz, p, p]),
        "yr_eval_topk_metrics_tc_slice": (C.c_int, [p, i64, p, p, i64, i64, i32, p, i64, p, p, p, p, p, p, i32,
                                                    p, p, p, p, p, sz, p, i32, i32, p, p]),
        "yr_recommend_ws_bytes": (sz, [i64, i64, i32]),
        "yr_recommend_topk": (C.c_int, [p, i64, p, i64, i32, i32, p, i64, p, p, i32, f32, i32, p, p, p, sz, p, p]),
        "yr_recommend_subset_ws_bytes": (sz, [i64, i32, i64, i32]),
        "yr_recommend_subset_topk": (C.c_int, [p, i64, p, i64, i32, i32, p, i64, p, p, i32, i64, p, p, p, i32, p, p, p,
                                               sz, p, p]),
        "yr_recommend_topk_ex": (C.c_int, [p, i64, p, i64, i32, i32, p, i64, p, p, i32, f32, i32, p, p, p, sz, p, p, p]),
        "yr_recommend_subset_topk_ex": (C.c_int, [p, i64, p, i64, i32, i32, p, i64, p, p, i32, i64, p, p, p, i32, p, p,
                                                  p, sz, p, p, p]),
        "yr_cdae_encode": (C.c_int, [C.POINTER(YrCdaeTensors), i64, i64, i32, i32, p, i64, p, p, p, i64, p, p]),
        "yr_recommend_geo_ws_bytes": (sz, [i64, i64, i32]),
        "yr_recommend_geo_topk": (C.c_int, [p, i64, p, i64, i32, i32, p, i64, p, p, i64, p, p, C.c_double, i64, i64, p,
                                            p, p, p, i32, p, p, p, sz, p, p, p]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc == 0:
        return
    if rc >= 1000:
        raise YelprecError(f"{what}: {_STATUS.get(rc, rc)}")
    raise YelprecError(f"{what}: cudaError {rc}")


def stream_ptr(device=None) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def dptr(t: Optional[torch.Tensor], dtype: Optional[torch.dtype] = None) -> Optional[int]:
    """Device pointer of a contiguous CUDA tensor (None passes through as NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise YelprecError("expected a CUDA tensor (the B200 path has no CPU fallback)")
    if not t.is_contiguous():
        raise YelprecError("expected a contiguous tensor")
    if dtype is not None and t.dtype != dtype:
        raise YelprecError(f"expected dtype {dtype}, got {t.dtype}")
    return t.data_ptr()


def make_opt(kind: str, lr: float, weight_decay: float = 0.0, step: int = 1,
             betas=(0.9, 0.999), eps: float = 1e-8) -> YrOpt:
    k = OPT_KINDS.get(str(kind).lower())
    if k is None:
        # reference: trainers/base_trainer.py:41-43
        raise NotImplementedError(f"Optimizer Not Exists: {kind}")
    return YrOpt(k, int(step), float(lr), float(weight_decay), float(betas[0]), float(betas[1]), float(eps))
