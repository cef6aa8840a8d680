"""ctypes binding of libb200rec.so (the C-ABI in include/b200rec.h).  No fallback: a missing library raises."""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# B200REC_LIB (development only): load a variant build of the same library for interleaved A/B timing
LIB_PATH = os.environ.get("B200REC_LIB") or os.path.join(_HERE, "libb200rec.so")

_lib = None

_P = C.c_void_p
_I64 = C.c_int64
_I = C.c_int
_F = C.c_float
_SZ = C.c_size_t
_U64 = C.c_uint64

# name -> (restype, argtypes); one entry per symbol declared in include/b200rec.h
_D = C.c_double
SIGNATURES = {
    "b200rec_last_error": (C.c_char_p, []),
    "b200rec_version": (_I, []),
    "b200rec_launch_count": (_I64, []),
    "b200rec_split_bf16": (_I, [_P, _I64, _I64, _I64, _I, _P, _I64, _I, _I, _P]),
    "b200rec_normalize_rows": (_I, [_P, _I64, _I64, _I64, _I, _I, _P, _I64, _P, _P, _I64, _I, _I, _P]),
    "b200rec_gemm_bf16_tn": (_I, [_P, _I64, _I64, _P, _I64, _I64, _I64, _P, _I64, _P, _F, _I, _P]),
    "b200rec_topk_workspace_bytes": (_SZ, [_I64, _I64, _I64, _I]),
    "b200rec_flat_ip_topk": (_I, [_P, _I64, _I64, _P, _I64, _I, _I64, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "b200rec_flat_ip_topk_filtered": (_I, [_P, _I64, _I64, _P, _I64, _I, _I64, _P, _I64, _P, _P, _P, _SZ, _P]),
    "b200rec_rows_to_bitmap": (_I, [_P, _I64, _I64, _P, _P]),
    "b200rec_remap_ids": (_I, [_P, _I64, _P, _I64, _I64, _P, _P]),
    "b200rec_update_rows": (_I, [_P, _I64, _I64, _I64, _I, _P, _I64, _P, _I64, _P, _I64, _I, _I, _P, _P]),
    "b200rec_clear_row_bits": (_I, [_P, _I64, _I64, _P, _P]),
    "b200rec_patch_compacted": (_I, [_P, _I64, _P, _I64, _P, _I64, _P, _P, _I, _P]),
    "b200rec_flat_ip_topk_masked": (_I, [_P, _I64, _I64, _P, _I64, _I, _I64, _P, _P, _P, _I64, _P, _I64, _P, _P, _P, _P,
                                         _SZ, _P]),
    "b200rec_topk_sample": (_I, [_P, _I64, _I64, _P, _I64, _I, _I, _I, _P, _P, _SZ, _P]),
    "b200rec_topk_has_sample": (_I, [_I64, _I64, _I64, _I]),
    "b200rec_topk_pooled_kth": (_I, [_P, _I, _I64, _I, _I, _P, _P]),
    "b200rec_flat_ip_topk_fanout": (_I, [_P, _I64, _I64, _P, _I64, _I, _I64, _P, _I, _P, _P, _P, _SZ, _P]),
    "b200rec_topk_sample_fanout": (_I, [_P, _I64, _I64, _P, _I64, _I, _I, _I, _I, _P, _P, _SZ, _P]),
    "b200rec_topk_sample_filtered": (_I, [_P, _I64, _I64, _P, _I64, _I, _I, _I, _P, _I64, _P, _P, _SZ, _P]),
    "b200rec_topk_sample_filtered_fanout": (_I, [_P, _I64, _I64, _P, _I64, _I, _I, _I, _P, _I64, _I, _P, _P, _SZ, _P]),
    "b200rec_flat_ip_topk_filtered_fanout": (_I, [_P, _I64, _I64, _P, _I64, _I, _I64, _P, _I64, _P, _I64, _P, _I, _P, _P,
                                                  _P, _SZ, _P]),
    "b200rec_flat_ip_topk_masked_fanout": (_I, [_P, _I64, _I64, _P, _I64, _I, _I64, _P, _I64, _P, _I64, _P, _I, _P, _P,
                                                _P, _SZ, _P]),
    "b200rec_topk_merge": (_I, [_P, _P, _I, _I64, _I, _I, _I64, _I64, _P, _P, _P]),
    "b200rec_rescore_fp32": (_I, [_P, _I64, _P, _I64, _I64, _I64, _I, _P, _I64, _I, _P, _P]),
    "b200rec_mlp_forward": (_I, [_P, _I64, _P, _P, _I64, _P, _I64, _I, _I, _I, _P, _I64, _I, _P, _I, _P, _P]),
    "b200rec_mlp_dgrad": (_I, [_P, _I64, _P, _P, _P, _I64, _I64, _I, _I, _I, _P, _I64, _P, _P, _P]),
    "b200rec_mlp_wgrad": (_I, [_P, _I64, _P, _P, _P, _P, _I64, _P, _I64, _I, _I, _I, _P, _I64, _P, _P, _P, _P]),
    "b200rec_gather_concat": (_I, [_P, _I64, _I64, _P, _P, _P, _P, _P, _P, _I, _I64, _P, _I64, _P, _P]),
    "b200rec_train_step_begin": (_I, [_P, _P, _F, _F, _P, _U64, _P]),
    "b200rec_adam_dense_dev": (_I, [_P, _P, _P, _P, _I64, _F, _F, _F, _F, _P, _P, _I, _P]),
    "b200rec_sparse_adam_dev": (_I, [_P, _P, _P, _I64, _I, _P, _P, _P, _I64, _F, _F, _F, _P, _P, _P]),
    "b200rec_gather_rows": (_I, [_P, _I64, _I, _I64, _P, _I64, _P, _I64, _P, _P]),
    "b200rec_sample_negatives": (_I, [_P, _I64, _P, _P, _I64, _I64, _I, _U64, _U64, _P, _P, _P]),
    "b200rec_sparse_grad_workspace_bytes": (_SZ, [_I64]),
    "b200rec_embedding_sparse_grad": (_I, [_P, _I64, _P, _I64, _I, _I64, _I64, _P, _P, _P, _P, _SZ, _P]),
    "b200rec_scatter_add_rows": (_I, [_P, _I64, _P, _I64, _I, _I64, _I64, _P, _I64, _P]),
    "b200rec_peer_allreduce_bytes": (_SZ, [_I]),
    "b200rec_peer_allreduce_f64": (_I, [_P, _I, _I, _I, _P, _I, _P, _P]),
    "b200rec_sparse_claim_accumulate": (_I, [_P, _I64, _P, _I64, _I, _I64, _I64, _P, _P, _P, _P]),
    "b200rec_scatter_add_rows_flagged": (_I, [_P, _I64, _P, _I64, _I, _I64, _I64, _P, _I64, _P, _P]),
    "b200rec_table_sumsq": (_I, [_P, _I64, _I64, _I, _P, _P, _P]),
    "b200rec_adam_table": (_I, [_P, _P, _P, _P, _I64, _I64, _I, _P, _F, _F, _F, _F, _F, _F, _F, _P, _P, _I, _P]),
    "b200rec_scatter_rows": (_I, [_P, _P, _P, _I64, _I, _P, _I64, _I, _P]),
    "b200rec_bn_forward": (_I, [_P, _I64, _I64, _I64, _I, _I, _F, _F, _P, _P, _P, _P, _F, _U64, _P, _P, _P, _I64, _P,
                                _P]),
    "b200rec_bn_backward": (_I, [_P, _I64, _P, _I64, _I64, _I64, _I, _I, _P, _P, _P, _F, _U64, _P, _I64, _P, _P, _P,
                                 _P, _P]),
    "b200rec_bn_forward_dp": (_I, [_P, _I64, _I64, _I64, _I, _F, _F, _P, _P, _P, _P, _F, _U64, _P, _P, _P, _I64, _P, _I,
                                   _I64, _P]),
    "b200rec_bn_backward_dp": (_I, [_P, _I64, _P, _I64, _I64, _I64, _I, _P, _P, _P, _F, _U64, _P, _I64, _P, _P, _P, _P,
                                    _I, _I64, _P]),
    "b200rec_act_dropout": (_I, [_P, _I64, _I64, _I64, _I, _F, _U64, _P, _I64, _P]),
    "b200rec_act_dropout_bwd": (_I, [_P, _I64, _P, _I64, _I64, _I64, _I, _F, _U64, _P, _I64, _P]),
    "b200rec_colsum": (_I, [_P, _I64, _I64, _I64, _P, _I, _P, _P]),
    "b200rec_normalize_bwd": (_I, [_P, _P, _P, _I64, _I64, _P, _P]),
    "b200rec_inbatch_lse_workspace_bytes": (_SZ, [_I64, _I64, _I64]),
    "b200rec_inbatch_lse": (_I, [_P, _P, _I64, _I64, _I64, _F, _P, _P, _SZ, _P]),
    "b200rec_lse_rows": (_I, [_P, _I64, _I64, _I64, _F, _I64, _P, _P, _P]),
    "b200rec_softmax_grad": (_I, [_P, _I64, _I64, _I64, _F, _P, _I64, _F, _P, _P, _I64, _P]),
    "b200rec_ce_sum": (_I, [_P, _P, _I64, _P, _P]),
    "b200rec_explicit_ce": (_I, [_P, _P, _P, _I64, _I64, _I64, _F, _P, _P, _P, _F, _P, _P, _P, _P, _P, _P]),
    "b200rec_rowdot": (_I, [_P, _P, _I64, _I64, _F, _P, _P, _P, _P]),
    "b200rec_rowdot_bwd": (_I, [_P, _P, _P, _I64, _I64, _F, _P, _P, _P]),
    "b200rec_sumsq": (_I, [_P, _I64, _P, _P]),
    "b200rec_clip_coef": (_I, [_P, _F, _P, _P, _P]),
    "b200rec_adam_dense": (_I, [_P, _P, _P, _P, _I64, _F, _F, _F, _F, _F, _F, _F, _P, _I, _P]),
    "b200rec_inbatch_grad_supported": (_I, [_I64, _I64, _I, _I, _I]),
    "b200rec_inbatch_grad": (_I, [_P, _I64, _P, _P, _I64, _P, _P, _I64, _P, _P, _I64, _P, _I64, _I64, _I, _I, _I, _F, _P, _I64,
                                  _F, _P, _P, _I64, _P, _I64, _P]),
    "b200rec_eval_metrics": (_I, [_P, _I64, _I, _I64, _P, _I64, _P, _P, _P, _P, _I, _P, _P, _P, _P, _P, _I64, _I, _P, _P]),
    "b200rec_sparse_adam": (_I, [_P, _P, _P, _I64, _I, _P, _P, _P, _I64, _F, _F, _F, _F, _F, _F, _P, _P]),
}


class BnBlock(C.Structure):
    """b200rec_bn_block (include/b200rec.h)."""
    _fields_ = [("z", _P), ("ldz", _I64), ("H", C.c_int32), ("act", C.c_int32), ("training", C.c_int32),
                ("update_running", C.c_int32), ("sums", _P), ("gamma", _P), ("beta", _P), ("running_mean", _P),
                ("running_var", _P), ("num_batches_tracked", _P), ("eps", _F), ("momentum", _F), ("drop_p", _F),
                ("seed", _U64), ("B_stat", _I64)]


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU or PyTorch fallback for the b200rec kernels)")
        _lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(_lib, name)
            fn.restype = res
            fn.argtypes = args
    return _lib


def last_error() -> str:
    return lib().b200rec_last_error().decode()


def check(rc: int, what: str) -> None:
    if rc != 0:
        raise RuntimeError(f"b200rec {what} failed: {last_error()}")


def launch_count() -> int:
    return int(lib().b200rec_launch_count())


def ptr(t):
    """device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    assert t.is_cuda, "b200rec kernels take CUDA tensors only"
    return t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream


def pad64(n: int) -> int:
    return (n + 63) // 64 * 64
