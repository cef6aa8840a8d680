"""Tensor-level wrappers over the C-ABI (include/b200rec.h).  Every function launches hand-written sm_100a kernels
asynchronously on torch's current CUDA stream; torch is used only to own device memory."""
from __future__ import annotations

import math
from typing import Optional, Tuple

import torch

from . import _native as N

BF16 = torch.bfloat16


def _f32c(t: torch.Tensor) -> torch.Tensor:
    if t.dtype != torch.float32:
        t = t.float()
    return t if t.is_contiguous() else t.contiguous()


# ------------------------------------------------------------------------------------------------ operand preparation
def split_bf16(x: torch.Tensor, terms: int = 1, side: int = 0, transpose: bool = False,
               kpad: Optional[int] = None) -> torch.Tensor:
    """fp32 [R, C] -> bf16 operand [R, terms*kpad] (or of x^T when transpose)."""
    assert x.dim() == 2 and x.dtype == torch.float32 and x.stride(1) == 1
    r, c = x.shape
    rows, cols = (c, r) if transpose else (r, c)
    kp = N.pad64(cols) if kpad is None else kpad
    out = torch.empty((rows, terms * kp), dtype=BF16, device=x.device)
    N.check(N.lib().b200rec_split_bf16(N.ptr(x), rows, cols, x.stride(0), int(transpose), N.ptr(out), kp, terms, side,
                                       N.stream()), "split_bf16")
    return out


def normalize_rows(x: torch.Tensor, normalize: bool = True, faiss_rule: bool = False, want_f32: bool = True,
                   want_norms: bool = False, terms: int = 0, side: int = 0):
    """Row L2 normalisation fused with the operand cast.  Returns (y_f32 | None, norms | None, y_bf16 | None)."""
    assert x.dim() == 2 and x.dtype == torch.float32 and x.stride(1) == 1
    r, c = x.shape
    y = torch.empty((r, c), dtype=torch.float32, device=x.device) if want_f32 else None
    nr = torch.empty((r,), dtype=torch.float32, device=x.device) if want_norms else None
    kp = N.pad64(c)
    yb = torch.empty((r, terms * kp), dtype=BF16, device=x.device) if terms else None
    N.check(N.lib().b200rec_normalize_rows(N.ptr(x), r, c, x.stride(0), int(normalize), int(faiss_rule), N.ptr(y),
                                           c, N.ptr(nr), N.ptr(yb), kp, max(terms, 1), side, N.stream()),
            "normalize_rows")
    return y, nr, yb


# ------------------------------------------------------------------------------------------------ GEMM
def gemm_tn(a_op: torch.Tensor, b_op: torch.Tensor, M: int, Nn: int, K: int, bias: Optional[torch.Tensor] = None,
            alpha: float = 1.0, k_splits: int = 1, out: Optional[torch.Tensor] = None,
            accumulate: bool = False) -> torch.Tensor:
    """C[M,N] = alpha * A[M,K] . B[N,K]^T + bias, bf16 operands, fp32 result.  accumulate=True adds into `out`
    (needs k_splits >= 2: the split-K path accumulates with fp32 atomics)."""
    assert a_op.dtype == BF16 and b_op.dtype == BF16
    if accumulate:
        assert out is not None and k_splits >= 2
    elif out is None:
        out = (torch.zeros if k_splits > 1 else torch.empty)((M, Nn), dtype=torch.float32, device=a_op.device)
    elif k_splits > 1:
        out.zero_()
    N.check(N.lib().b200rec_gemm_bf16_tn(N.ptr(a_op), a_op.stride(0), M, N.ptr(b_op), b_op.stride(0), Nn, K,
                                         N.ptr(out), out.stride(0), N.ptr(bias), float(alpha), -k_splits if accumulate else k_splits,
                                         N.stream()),
            "gemm_bf16_tn")
    return out


def matmul_nt(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None, terms: int = 6,
              k_splits: int = 1) -> torch.Tensor:
    """x[M,K] . w[N,K]^T (+bias) through split-bf16 operands (terms=6: fp32-grade; 1: plain bf16)."""
    xo = split_bf16(_f32c(x), terms, 0)
    wo = split_bf16(_f32c(w), terms, 1)
    return gemm_tn(xo, wo, x.shape[0], w.shape[0], xo.shape[1], bias, 1.0, k_splits)


# ------------------------------------------------------------------------------------------------ exact IP top-K
def topk_workspace_bytes(n: int, ld: int, q: int, k: int) -> int:
    return int(N.lib().b200rec_topk_workspace_bytes(n, ld, q, k))


def flat_ip_topk(catalogue: torch.Tensor, queries: torch.Tensor, k: int, row_offset: int = 0,
                 exclude_indptr: Optional[torch.Tensor] = None, exclude_rows: Optional[torch.Tensor] = None,
                 workspace: Optional[torch.Tensor] = None, tau_init: Optional[torch.Tensor] = None,
                 out: Optional[Tuple[torch.Tensor, torch.Tensor]] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """catalogue bf16 [N, ld], queries bf16 [Q, ld] (ld multiple of 64) -> (scores fp32 [Q,k] desc, ids int64 [Q,k])."""
    assert catalogue.dtype == BF16 and queries.dtype == BF16
    assert catalogue.stride(1) == 1 and queries.stride(1) == 1 and catalogue.stride(0) == queries.stride(0)
    n, ld = catalogue.shape[0], catalogue.stride(0)
    q = queries.shape[0]
    need = topk_workspace_bytes(n, ld, q, k)
    if need == 0:
        raise RuntimeError(f"b200rec flat_ip_topk: {N.last_error()}")
    if workspace is None or workspace.numel() < need:
        workspace = torch.empty((need,), dtype=torch.uint8, device=catalogue.device)
    if out is None:
        scores = torch.empty((q, k), dtype=torch.float32, device=catalogue.device)
        ids = torch.empty((q, k), dtype=torch.int64, device=catalogue.device)
    else:
        scores, ids = out
    N.check(N.lib().b200rec_flat_ip_topk(N.ptr(catalogue), n, ld, N.ptr(queries), q, k, row_offset,
                                         N.ptr(exclude_indptr), N.ptr(exclude_rows), N.ptr(tau_init), N.ptr(scores),
                                         N.ptr(ids), N.ptr(workspace), workspace.numel(), N.stream()), "flat_ip_topk")
    return scores, ids


def flat_ip_topk_filtered(catalogue: torch.Tensor, queries: torch.Tensor, k: int, allow_bits: torch.Tensor,
                          allow_n: int, row_offset: int = 0, workspace: Optional[torch.Tensor] = None
                          ) -> Tuple[torch.Tensor, torch.Tensor]:
    """flat_ip_topk over the rows allowed by a bitmap (int32/uint32 words, bit r of word r >> 5; rows >= allow_n out)."""
    assert catalogue.dtype == BF16 and queries.dtype == BF16 and allow_bits.dtype == torch.int32
    assert catalogue.stride(1) == 1 and queries.stride(1) == 1 and catalogue.stride(0) == queries.stride(0)
    n, ld = catalogue.shape[0], catalogue.stride(0)
    q = queries.shape[0]
    assert allow_bits.numel() * 32 >= min(allow_n, n)
    need = topk_workspace_bytes(n, ld, q, k)
    if need == 0:
        raise RuntimeError(f"b200rec flat_ip_topk_filtered: {N.last_error()}")
    if workspace is None or workspace.numel() < need:
        workspace = torch.empty((need,), dtype=torch.uint8, device=catalogue.device)
    scores = torch.empty((q, k), dtype=torch.float32, device=catalogue.device)
    ids = torch.empty((q, k), dtype=torch.int64, device=catalogue.device)
    N.check(N.lib().b200rec_flat_ip_topk_filtered(N.ptr(catalogue), n, ld, N.ptr(queries), q, k, row_offset,
                                                  N.ptr(allow_bits), allow_n, N.ptr(scores), N.ptr(ids),
                                                  N.ptr(workspace), workspace.numel(), N.stream()), "flat_ip_topk_filtered")
    return scores, ids


def rows_to_bitmap(rows: torch.Tensor, n_bits: int) -> torch.Tensor:
    """int64 rows -> int32 [ceil(n_bits / 32)] bitmap (faiss IDSelectorBitmap layout); rows outside [0, n_bits) ignored."""
    assert rows.dtype == torch.int64 and rows.is_contiguous()
    bits = torch.empty(((n_bits + 31) // 32,), dtype=torch.int32, device=rows.device)
    N.check(N.lib().b200rec_rows_to_bitmap(N.ptr(rows), rows.numel(), n_bits, N.ptr(bits), N.stream()), "rows_to_bitmap")
    return bits


def remap_ids(ids: torch.Tensor, rows: torch.Tensor, row_offset: int = 0) -> torch.Tensor:
    """ids of a search over catalogue rows `rows` (ascending) -> rows[ids] + row_offset, in place; -1 stays -1."""
    assert ids.dtype == torch.int64 and ids.is_contiguous() and rows.dtype == torch.int64 and rows.is_contiguous()
    N.check(N.lib().b200rec_remap_ids(N.ptr(ids), ids.numel(), N.ptr(rows), rows.numel(), row_offset, N.ptr(ids),
                                      N.stream()), "remap_ids")
    return ids


def topk_pooled_kth(vals: torch.Tensor, k: int) -> torch.Tensor:
    """vals [parts, Q, k_in] fp32 (contiguous) -> [Q]: k-th largest of each query's parts*k_in pooled sample maxima."""
    assert vals.dim() == 3 and vals.is_contiguous() and vals.dtype == torch.float32
    parts, q, k_in = vals.shape
    out = torch.empty((q,), dtype=torch.float32, device=vals.device)
    N.check(N.lib().b200rec_topk_pooled_kth(N.ptr(vals), parts, q, k_in, k, N.ptr(out), N.stream()), "topk_pooled_kth")
    return out


def _ptr_table(ptrs):
    import ctypes
    return (ctypes.c_void_p * len(ptrs))(*[int(p) for p in ptrs])


def flat_ip_topk_fanout(catalogue: torch.Tensor, queries: torch.Tensor, k: int, row_offset: int,
                        tau_init: Optional[torch.Tensor], dst_scores, dst_ids, workspace: torch.Tensor) -> None:
    """flat_ip_topk whose [Q,k] result rows are stored to every (dst_scores[d], dst_ids[d]) device address — this shard's
    slot in each GPU's gather buffer (peer-mapped symmetric memory): the select kernel doubles as the all-gather."""
    n, ld, q = catalogue.shape[0], catalogue.stride(0), queries.shape[0]
    N.check(N.lib().b200rec_flat_ip_topk_fanout(N.ptr(catalogue), n, ld, N.ptr(queries), q, k, row_offset,
                                                N.ptr(tau_init), len(dst_scores), _ptr_table(dst_scores),
                                                _ptr_table(dst_ids), N.ptr(workspace), workspace.numel(), N.stream()),
            "flat_ip_topk_fanout")


def topk_sample_fanout(catalogue: torch.Tensor, queries: torch.Tensor, k: int, k_out: int, shards: int, dst_vals,
                       workspace: torch.Tensor) -> None:
    n, ld, q = catalogue.shape[0], catalogue.stride(0), queries.shape[0]
    N.check(N.lib().b200rec_topk_sample_fanout(N.ptr(catalogue), n, ld, N.ptr(queries), q, k, k_out, shards,
                                               len(dst_vals), _ptr_table(dst_vals), N.ptr(workspace),
                                               workspace.numel(), N.stream()), "topk_sample_fanout")


def topk_sample_filtered(catalogue: Optional[torch.Tensor], queries: torch.Tensor, k: int, k_out: int, shards: int,
                         allow_bits: Optional[torch.Tensor], allow_n: int, workspace: Optional[torch.Tensor],
                         dst_vals=None) -> Optional[torch.Tensor]:
    """Sampling pass of one row shard of a filtered search: the k_out largest group maxima per query over the rows the
    bitmap allows (allow_bits None: every row of `catalogue`, a compacted one).  -FLT_MAX rows when nothing is allowed or
    the shape has no sampling pass.  dst_vals (device addresses): stored to every one of them, else returned [Q, k_out].
    catalogue / workspace may be None when the shard holds no row."""
    n = 0 if catalogue is None else catalogue.shape[0]
    ld = queries.stride(0)
    q = queries.shape[0]
    ws_n = 0 if workspace is None else workspace.numel()
    if dst_vals is None:
        vals = torch.empty((q, k_out), dtype=torch.float32, device=queries.device)
        N.check(N.lib().b200rec_topk_sample_filtered(N.ptr(catalogue), n, ld, N.ptr(queries), q, k, k_out, shards,
                                                     N.ptr(allow_bits), allow_n, N.ptr(vals), N.ptr(workspace), ws_n,
                                                     N.stream()), "topk_sample_filtered")
        return vals
    N.check(N.lib().b200rec_topk_sample_filtered_fanout(N.ptr(catalogue), n, ld, N.ptr(queries), q, k, k_out, shards,
                                                        N.ptr(allow_bits), allow_n, len(dst_vals), _ptr_table(dst_vals),
                                                        N.ptr(workspace), ws_n, N.stream()), "topk_sample_filtered_fanout")
    return None


def flat_ip_topk_filtered_fanout(catalogue: Optional[torch.Tensor], queries: torch.Tensor, k: int, row_offset: int,
                                 allow_bits: Optional[torch.Tensor], allow_n: int, remap_rows: Optional[torch.Tensor],
                                 tau_init: Optional[torch.Tensor], dst_scores, dst_ids,
                                 workspace: Optional[torch.Tensor]) -> None:
    """Local top-k of one row shard of a filtered search, from tau_init, stored to every (dst_scores[d], dst_ids[d]).
    Exactly one of allow_bits (bitmap over `catalogue`) and remap_rows (int64: `catalogue` is compacted, its row j is local
    row remap_rows[j]; the select kernel stores remap_rows[j] + row_offset) is given.  -1 / -FLT_MAX rows when nothing is
    allowed; catalogue / workspace may then be None."""
    n = 0 if catalogue is None else catalogue.shape[0]
    n_remap = 0 if remap_rows is None else remap_rows.numel()
    N.check(N.lib().b200rec_flat_ip_topk_filtered_fanout(N.ptr(catalogue), n, queries.stride(0), N.ptr(queries),
                                                         queries.shape[0], k, row_offset, N.ptr(allow_bits), allow_n,
                                                         N.ptr(remap_rows), n_remap, N.ptr(tau_init), len(dst_scores),
                                                         _ptr_table(dst_scores), _ptr_table(dst_ids), N.ptr(workspace),
                                                         0 if workspace is None else workspace.numel(), N.stream()),
            "flat_ip_topk_filtered_fanout")


def topk_has_sample(n: int, ld: int, q: int, k: int) -> bool:
    return bool(N.lib().b200rec_topk_has_sample(n, ld, q, k))


def topk_sample(catalogue: torch.Tensor, queries: torch.Tensor, k: int, workspace: torch.Tensor,
                k_out: Optional[int] = None, shards: int = 1) -> torch.Tensor:
    """Sampling pass only: [Q,k_out] largest group maxima per query (what row shards exchange before the main pass).
    `shards` row shards pool their samples, so each samples 1/shards as densely."""
    n, ld, q = catalogue.shape[0], catalogue.stride(0), queries.shape[0]
    k_out = k if k_out is None else k_out
    vals = torch.empty((q, k_out), dtype=torch.float32, device=catalogue.device)
    N.check(N.lib().b200rec_topk_sample(N.ptr(catalogue), n, ld, N.ptr(queries), q, k, k_out, shards, N.ptr(vals),
                                        N.ptr(workspace), workspace.numel(), N.stream()), "topk_sample")
    return vals


def topk_merge(scores: torch.Tensor, ids: torch.Tensor, k_out: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """scores/ids [parts, Q, k_in] -> global top k_out per query (score desc, id asc; id < 0 = padding).  The part
    dimension may be strided (scores and ids interleaved in one all-gathered buffer)."""
    assert scores.dim() == 3 and scores.shape == ids.shape
    parts, q, k_in = scores.shape
    assert scores.stride(2) == 1 and scores.stride(1) == k_in and ids.stride(2) == 1 and ids.stride(1) == k_in
    out_s = torch.empty((q, k_out), dtype=torch.float32, device=scores.device)
    out_i = torch.empty((q, k_out), dtype=torch.int64, device=scores.device)
    N.check(N.lib().b200rec_topk_merge(N.ptr(scores), N.ptr(ids), parts, q, k_in, k_out, scores.stride(0),
                                       ids.stride(0), N.ptr(out_s), N.ptr(out_i), N.stream()), "topk_merge")
    return out_s, out_i


def rescore_fp32(queries: torch.Tensor, rows: torch.Tensor, ids: torch.Tensor, row_offset: int = 0) -> torch.Tensor:
    """Exact fp32 inner products of candidate rows: queries fp32 [Q, d], rows fp32 [n, d], ids int64 [Q, k_in] (global
    ids, < 0 = empty) -> scores fp32 [Q, k_in] (-FLT_MAX at empty slots)."""
    assert queries.dtype == torch.float32 and rows.dtype == torch.float32 and ids.dtype == torch.int64
    assert queries.stride(1) == 1 and rows.stride(1) == 1 and ids.is_contiguous()
    q, k_in = ids.shape
    out = torch.empty((q, k_in), dtype=torch.float32, device=ids.device)
    N.check(N.lib().b200rec_rescore_fp32(N.ptr(queries), queries.stride(0), N.ptr(rows), rows.stride(0), rows.shape[0],
                                         row_offset, queries.shape[1], N.ptr(ids), q, k_in, N.ptr(out), N.stream()),
            "rescore_fp32")
    return out


# ------------------------------------------------------------------------------------------------ embedding bags
import ctypes as _C  # noqa: E402


def gather_concat(numerical: Optional[torch.Tensor], tables, indices, widths, col_offsets, out_cols: int,
                  batch: int, device, err: torch.Tensor) -> torch.Tensor:
    """Fused multi-field gather writing the MLP input [B, out_cols] (numerical block first).  `err` (int32[1]) is set to
    field + 1 when an id lies outside its table (ops.check_index_errors raises IndexError from it)."""
    F = len(tables)
    out = torch.empty((batch, out_cols), dtype=torch.float32, device=device)
    num_cols = 0 if numerical is None else numerical.shape[1]
    tp = (_C.c_void_p * max(F, 1))(*[t.data_ptr() for t in tables])
    ip = (_C.c_void_p * max(F, 1))(*[i.data_ptr() for i in indices])
    rows = (_C.c_int64 * max(F, 1))(*[t.shape[0] for t in tables])
    wd = (_C.c_int32 * max(F, 1))(*widths)
    tld = (_C.c_int32 * max(F, 1))(*[t.stride(0) for t in tables])
    co = (_C.c_int32 * max(F, 1))(*col_offsets)
    N.check(N.lib().b200rec_gather_concat(N.ptr(numerical), num_cols, numerical.stride(0) if numerical is not None else 0,
                                          tp, ip, rows, wd, tld, co, F, batch, N.ptr(out), out.stride(0), N.ptr(err),
                                          N.stream()), "gather_concat")
    return out


def embedding_sparse_grad(idx: torch.Tensor, dY: torch.Tensor, width: int, table_rows: int, padding_idx: int = 0):
    """dY: [B, >=width] view (column block of the concat gradient).  Returns (rows int64 [B], grads [B,width], n int32[1]);
    only the first n entries are valid."""
    B = idx.shape[0]
    rows = torch.empty((B,), dtype=torch.int64, device=idx.device)
    grads = torch.empty((B, width), dtype=torch.float32, device=idx.device)
    n = torch.zeros((1,), dtype=torch.int32, device=idx.device)
    ws_bytes = int(N.lib().b200rec_sparse_grad_workspace_bytes(B))
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=idx.device)
    N.check(N.lib().b200rec_embedding_sparse_grad(N.ptr(idx), B, N.ptr(dY), dY.stride(0), width, padding_idx,
                                                  table_rows, N.ptr(rows), N.ptr(grads), N.ptr(n), N.ptr(ws), ws_bytes,
                                                  N.stream()), "embedding_sparse_grad")
    return rows, grads, n


def sparse_claim_accumulate(idx: torch.Tensor, dY: torch.Tensor, width: int, table_rows: int, slot: torch.Tensor,
                            padding_idx: int = 0):
    """Sort-free coalescing for row-sparse tables: returns (rows int64 [B] with -1 for duplicates / invalid ids,
    grads [B, width] with every distinct row's summed gradient in its leader's row, n int32[1] = B)."""
    B = idx.shape[0]
    rows = torch.empty((B,), dtype=torch.int64, device=idx.device)
    acc = torch.zeros((B, width), dtype=torch.float32, device=idx.device)
    n = torch.full((1,), B, dtype=torch.int32, device=idx.device)
    N.check(N.lib().b200rec_sparse_claim_accumulate(N.ptr(idx), B, N.ptr(dY), dY.stride(0), width, padding_idx, table_rows,
                                                    N.ptr(slot), N.ptr(rows), N.ptr(acc), N.stream()),
            "sparse_claim_accumulate")
    return rows, acc, n


def scatter_add_rows(idx: torch.Tensor, dY: torch.Tensor, width: int, dense: torch.Tensor, padding_idx: int = 0,
                     row_flags: Optional[torch.Tensor] = None) -> None:
    """dense[idx[b], :width] += dY[b, :width] with fp32 atomics (padding row and out-of-range ids skipped);
    row_flags (int32 [rows]): also raise the flag of every row that received a gradient."""
    if row_flags is not None:
        N.check(N.lib().b200rec_scatter_add_rows_flagged(N.ptr(idx), idx.shape[0], N.ptr(dY), dY.stride(0), width,
                                                         padding_idx, dense.shape[0], N.ptr(dense), dense.stride(0),
                                                         N.ptr(row_flags), N.stream()), "scatter_add_rows_flagged")
        return
    N.check(N.lib().b200rec_scatter_add_rows(N.ptr(idx), idx.shape[0], N.ptr(dY), dY.stride(0), width, padding_idx,
                                             dense.shape[0], N.ptr(dense), dense.stride(0), N.stream()), "scatter_add_rows")


def scatter_rows(rows, grads, n, dense: torch.Tensor, accumulate: bool = False) -> None:
    N.check(N.lib().b200rec_scatter_rows(N.ptr(rows), N.ptr(grads), N.ptr(n), rows.shape[0], grads.shape[1],
                                         N.ptr(dense), dense.stride(0), int(accumulate), N.stream()), "scatter_rows")


# ------------------------------------------------------------------------------------------------ tower pieces
ACT_IDS = {"relu": 0, "gelu": 1, "leaky_relu": 2, "tanh": 3, "sigmoid": 4, "identity": 5}


def _scratch(n_doubles: int, device) -> torch.Tensor:
    return torch.empty((n_doubles,), dtype=torch.float64, device=device)


def bn_forward(z, act: int, training: bool, eps: float, momentum: float, gamma, beta, running_mean, running_var,
               drop_p: float, seed: int):
    B, H = z.shape
    y = torch.empty_like(z)
    mean = torch.empty((H,), dtype=torch.float32, device=z.device)
    invstd = torch.empty((H,), dtype=torch.float32, device=z.device)
    N.check(N.lib().b200rec_bn_forward(N.ptr(z), B, H, z.stride(0), act, int(training), eps, momentum, N.ptr(gamma),
                                       N.ptr(beta), N.ptr(running_mean), N.ptr(running_var), drop_p, seed, N.ptr(mean),
                                       N.ptr(invstd), N.ptr(y), y.stride(0), N.ptr(_scratch(3 * H, z.device)),
                                       N.stream()), "bn_forward")
    return y, mean, invstd


def bn_backward(dy, z, act: int, training: bool, mean, invstd, gamma, drop_p: float, seed: int):
    B, H = z.shape
    dz = torch.empty_like(z)
    dgamma = torch.zeros((H,), dtype=torch.float32, device=z.device)
    dbeta = torch.zeros((H,), dtype=torch.float32, device=z.device)
    N.check(N.lib().b200rec_bn_backward(N.ptr(dy), dy.stride(0), N.ptr(z), z.stride(0), B, H, act, int(training),
                                        N.ptr(mean), N.ptr(invstd), N.ptr(gamma), drop_p, seed, N.ptr(dz), dz.stride(0),
                                        N.ptr(dgamma), N.ptr(dbeta), None, N.ptr(_scratch(3 * H, z.device)),
                                        N.stream()), "bn_backward")
    return dz, dgamma, dbeta


def bn_forward_dp(z, act: int, eps: float, momentum: float, gamma, beta, running_mean, running_var, drop_p: float,
                  seed: int, reduce_sums, b_total: int):
    """Training-mode BatchNorm with statistics over all data-parallel replicas.  `reduce_sums(t)` all-reduces (sum) the
    fp64 tensor t in place (torch.distributed.all_reduce on the NCCL group)."""
    B, H = z.shape
    y = torch.empty_like(z)
    mean = torch.empty((H,), dtype=torch.float32, device=z.device)
    invstd = torch.empty((H,), dtype=torch.float32, device=z.device)
    scratch = _scratch(3 * H, z.device)
    args = (N.ptr(z), B, H, z.stride(0), act, eps, momentum, N.ptr(gamma), N.ptr(beta), N.ptr(running_mean),
            N.ptr(running_var), drop_p, seed, N.ptr(mean), N.ptr(invstd), N.ptr(y), y.stride(0), N.ptr(scratch))
    N.check(N.lib().b200rec_bn_forward_dp(*args, 0, b_total, N.stream()), "bn_forward_dp")
    reduce_sums(scratch[: 2 * H])
    N.check(N.lib().b200rec_bn_forward_dp(*args, 1, b_total, N.stream()), "bn_forward_dp")
    return y, mean, invstd


def bn_backward_dp(dy, z, act: int, mean, invstd, gamma, drop_p: float, seed: int, reduce_sums, b_total: int):
    B, H = z.shape
    dz = torch.empty_like(z)
    dgamma = torch.zeros((H,), dtype=torch.float32, device=z.device)
    dbeta = torch.zeros((H,), dtype=torch.float32, device=z.device)
    scratch = _scratch(3 * H, z.device)
    args = (N.ptr(dy), dy.stride(0), N.ptr(z), z.stride(0), B, H, act, N.ptr(mean), N.ptr(invstd), N.ptr(gamma), drop_p,
            seed, N.ptr(dz), dz.stride(0), N.ptr(dgamma), N.ptr(dbeta), None, N.ptr(scratch))
    N.check(N.lib().b200rec_bn_backward_dp(*args, 0, b_total, N.stream()), "bn_backward_dp")
    reduce_sums(scratch[: 2 * H])
    N.check(N.lib().b200rec_bn_backward_dp(*args, 1, b_total, N.stream()), "bn_backward_dp")
    return dz, dgamma, dbeta


# ------------------------------------------------------------------------------------------------ fused MLP layers
class BnBlock:
    """One hidden block [Linear -> act -> BatchNorm1d -> Dropout] as the fused layer kernels see it (b200rec_bn_block):
    the block's pre-activations z, its batch statistics (fp64 sums) or running statistics, affine and dropout stream."""

    def __init__(self, z, act: int, training: bool, sums, gamma, beta, running_mean, running_var, nbt, eps: float,
                 momentum: float, drop_p: float, seed: int, b_stat: int, update_running: bool = False):
        self.z, self.sums, self.gamma, self.beta = z, sums, gamma, beta
        self.running_mean, self.running_var, self.nbt = running_mean, running_var, nbt
        self.c = N.BnBlock(N.ptr(z), z.stride(0), z.shape[1], act, int(training), int(update_running), N.ptr(sums),
                           N.ptr(gamma), N.ptr(beta), N.ptr(running_mean), N.ptr(running_var), N.ptr(nbt), eps, momentum,
                           drop_p if training else 0.0, seed & 0xFFFFFFFFFFFFFFFF, b_stat)

    def ref(self, update_running: Optional[bool] = None):
        if update_running is not None:
            self.c.update_running = int(update_running)
        return _C.byref(self.c)


def mlp_forward(x: Optional[torch.Tensor], lower: Optional[BnBlock], w, bias, out: torch.Tensor, np_: int, out_act: int = 5,
                out_sums: Optional[torch.Tensor] = None, normalize: bool = False, norms: Optional[torch.Tensor] = None,
                update_running: bool = False) -> torch.Tensor:
    """out[B,N] = input . w^T + bias (input = x or the output of block `lower`), one launch (csrc/mlp_fused.cuh)."""
    B, Nn, Kk = out.shape[0], w.shape[0], w.shape[1]
    N.check(N.lib().b200rec_mlp_forward(N.ptr(x), x.stride(0) if x is not None else 0,
                                        lower.ref(update_running) if lower is not None else None, N.ptr(w), w.stride(0),
                                        N.ptr(bias), B, Nn, Kk, np_, N.ptr(out), out.stride(0), out_act, N.ptr(out_sums),
                                        int(normalize), N.ptr(norms), N.stream()), "mlp_forward")
    return out


def mlp_dgrad(dy, own: Optional[BnBlock], own_bsums, w, dx, np_: int, lower: Optional[BnBlock] = None,
              lower_bsums: Optional[torch.Tensor] = None) -> torch.Tensor:
    B, Nn, Kk = dy.shape[0], w.shape[0], w.shape[1]
    N.check(N.lib().b200rec_mlp_dgrad(N.ptr(dy), dy.stride(0), own.ref() if own is not None else None, N.ptr(own_bsums),
                                      N.ptr(w), w.stride(0), B, Nn, Kk, np_, N.ptr(dx), dx.stride(0),
                                      lower.ref() if lower is not None else None, N.ptr(lower_bsums), N.stream()),
            "mlp_dgrad")
    return dx


def mlp_wgrad(dy, own: Optional[BnBlock], own_bsums, own_bsums_local, x, lower: Optional[BnBlock], np_: int, dw, db,
              dgamma=None, dbeta=None) -> None:
    B, Nn, Kk = dy.shape[0], dw.shape[0], dw.shape[1]
    N.check(N.lib().b200rec_mlp_wgrad(N.ptr(dy), dy.stride(0), own.ref() if own is not None else None, N.ptr(own_bsums),
                                      N.ptr(own_bsums_local), N.ptr(x), x.stride(0) if x is not None else 0,
                                      lower.ref() if lower is not None else None, B, Nn, Kk, np_, N.ptr(dw), dw.stride(0),
                                      N.ptr(db), N.ptr(dgamma), N.ptr(dbeta), N.stream()), "mlp_wgrad")


def act_dropout(z, act: int, drop_p: float, seed: int):
    B, H = z.shape
    y = torch.empty_like(z)
    N.check(N.lib().b200rec_act_dropout(N.ptr(z), B, H, z.stride(0), act, drop_p, seed, N.ptr(y), y.stride(0),
                                        N.stream()), "act_dropout")
    return y


def act_dropout_bwd(dy, z, act: int, drop_p: float, seed: int):
    B, H = z.shape
    dz = torch.empty_like(z)
    N.check(N.lib().b200rec_act_dropout_bwd(N.ptr(dy), dy.stride(0), N.ptr(z), z.stride(0), B, H, act, drop_p, seed,
                                            N.ptr(dz), dz.stride(0), N.stream()), "act_dropout_bwd")
    return dz


def colsum(x) -> torch.Tensor:
    B, H = x.shape
    out = torch.empty((H,), dtype=torch.float32, device=x.device)
    N.check(N.lib().b200rec_colsum(N.ptr(x), B, H, x.stride(0), N.ptr(out), 0, N.ptr(_scratch(H, x.device)),
                                   N.stream()), "colsum")
    return out


def normalize_bwd(dE, E, norms):
    dE = _f32c(dE)
    dO = torch.empty_like(E)
    N.check(N.lib().b200rec_normalize_bwd(N.ptr(dE), N.ptr(E), N.ptr(norms), E.shape[0], E.shape[1], N.ptr(dO),
                                          N.stream()), "normalize_bwd")
    return dO


# ------------------------------------------------------------------------------------------------ losses
def inbatch_lse(u_op, i_op, B: int, NI: int, inv_t: float):
    """Fused logits GEMM + online log-sum-exp; returns None when the operand is too wide for the resident tile."""
    ld = u_op.stride(0)
    need = int(N.lib().b200rec_inbatch_lse_workspace_bytes(B, NI, ld))
    if need == 0:
        return None
    ws = torch.empty((need,), dtype=torch.uint8, device=u_op.device)
    lse = torch.empty((B,), dtype=torch.float32, device=u_op.device)
    N.check(N.lib().b200rec_inbatch_lse(N.ptr(u_op), N.ptr(i_op), ld, B, NI, inv_t, N.ptr(lse), N.ptr(ws), need,
                                        N.stream()), "inbatch_lse")
    return lse


# block index of pieces (h, m, l) inside an operand row written by split_bf16(terms, side) — csrc/prep.cu part_of()
PIECE_BLOCKS = {(1, 0): (0,), (1, 1): (0,), (3, 0): (0, 1), (3, 1): (1, 0), (6, 0): (2, 0, 1), (6, 1): (1, 0, 2)}


def inbatch_grad_supported(B: int, NI: int, E: int, nprod_s: int, nprod_g: int) -> bool:
    return bool(N.lib().b200rec_inbatch_grad_supported(B, NI, E, nprod_s, nprod_g))


def inbatch_grad(u_op, u_blocks, v_op, v_blocks, B: int, NI: int, E: int, nprod_s: int, nprod_g: int, inv_t: float, lse,
                 diag0: int, coef: float, coef_dev, dU, dV) -> None:
    """Fused in-batch loss backward (csrc/inbatch_grad.cu): logits recomputed tile-wise in TMEM, G = softmax - onehot
    formed in registers, both gradient GEMMs fed from shared memory (the row operands double as the MN-major operand of
    the gradient GEMMs: no transposed copies).  Writes dU [B,E] and dV [NI,E] completely."""
    def tab(blocks):
        b = list(blocks) + [0] * (3 - len(blocks))
        return (_C.c_int32 * 3)(*b)
    N.check(N.lib().b200rec_inbatch_grad(N.ptr(u_op), u_op.stride(0), tab(u_blocks), N.ptr(v_op), v_op.stride(0), tab(v_blocks),
                                         None, 0, None, None, 0, None, B, NI, E, nprod_s, nprod_g, float(inv_t), N.ptr(lse),
                                         int(diag0), float(coef), N.ptr(coef_dev), N.ptr(dU), dU.stride(0), N.ptr(dV),
                                         dV.stride(0), N.stream()), "inbatch_grad")


def lse_rows(S, scale: float, diag0: int, want_pos: bool):
    rows, cols = S.shape
    lse = torch.empty((rows,), dtype=torch.float32, device=S.device)
    pos = torch.empty((rows,), dtype=torch.float32, device=S.device) if want_pos else None
    N.check(N.lib().b200rec_lse_rows(N.ptr(S), S.stride(0), rows, cols, scale, diag0, N.ptr(lse), N.ptr(pos),
                                     N.stream()), "lse_rows")
    return lse, pos


def softmax_grad_(S, scale: float, lse, diag0: int, coef: float, coef_dev=None):
    rows, cols = S.shape
    N.check(N.lib().b200rec_softmax_grad(N.ptr(S), S.stride(0), rows, cols, scale, N.ptr(lse), diag0, coef,
                                         N.ptr(coef_dev), N.ptr(S), S.stride(0), N.stream()), "softmax_grad")
    return S


def ce_sum(lse, pos, acc) -> None:
    N.check(N.lib().b200rec_ce_sum(N.ptr(lse), N.ptr(pos), lse.shape[0], N.ptr(acc), N.stream()), "ce_sum")


def explicit_ce(U, P, Nn, R: int, inv_t: float, user_bias, item_bias, grad_scale: float = 0.0, grad_scale_dev=None,
                want_grad: bool = False):
    B, E = U.shape
    row_loss = torch.empty((B,), dtype=torch.float32, device=U.device)
    dU = dP = dN = dbias = None
    if want_grad:
        dU, dP, dN = torch.empty_like(U), torch.empty_like(P), torch.empty_like(Nn)
        dbias = torch.empty((B,), dtype=torch.float32, device=U.device)
    N.check(N.lib().b200rec_explicit_ce(N.ptr(U), N.ptr(P), N.ptr(Nn), B, R, E, inv_t, N.ptr(user_bias),
                                        N.ptr(item_bias), N.ptr(row_loss), grad_scale, N.ptr(grad_scale_dev), N.ptr(dU),
                                        N.ptr(dP), N.ptr(dN), N.ptr(dbias), N.stream()), "explicit_ce")
    return row_loss, dU, dP, dN, dbias


def rowdot(U, I, scale: float, user_bias, item_bias):
    B, E = U.shape
    out = torch.empty((B,), dtype=torch.float32, device=U.device)
    N.check(N.lib().b200rec_rowdot(N.ptr(U), N.ptr(I), B, E, scale, N.ptr(user_bias), N.ptr(item_bias), N.ptr(out),
                                   N.stream()), "rowdot")
    return out


def rowdot_bwd(g, U, I, scale: float):
    dU, dI = torch.empty_like(U), torch.empty_like(I)
    N.check(N.lib().b200rec_rowdot_bwd(N.ptr(g), N.ptr(U), N.ptr(I), U.shape[0], U.shape[1], scale, N.ptr(dU),
                                       N.ptr(dI), N.stream()), "rowdot_bwd")
    return dU, dI


# ------------------------------------------------------------------------------------------------ optimiser
def sumsq_(x_flat, acc64) -> None:
    N.check(N.lib().b200rec_sumsq(N.ptr(x_flat), x_flat.numel(), N.ptr(acc64), N.stream()), "sumsq")


def table_sumsq_(grad2d, row_flags, acc64) -> None:
    """acc64 += sum of squares of the flagged rows of a dense table gradient [rows, e]."""
    N.check(N.lib().b200rec_table_sumsq(N.ptr(grad2d), grad2d.stride(0), grad2d.shape[0], grad2d.shape[1], N.ptr(row_flags),
                                        N.ptr(acc64), N.stream()), "table_sumsq")


def adam_table_(p2d, g2d, m2d, v2d, row_flags, lr, beta1, beta2, eps, wd, step: int, clip=None, hyper_dev=None,
                clear_grad: bool = True) -> None:
    """Adam + L2-coupled weight decay over every row of a dense table, reading the gradient of flagged rows only."""
    bc1 = 1.0 - beta1 ** step if hyper_dev is None else 1.0
    bc2s = math.sqrt(1.0 - beta2 ** step) if hyper_dev is None else 1.0
    N.check(N.lib().b200rec_adam_table(N.ptr(p2d), N.ptr(g2d), N.ptr(m2d), N.ptr(v2d), p2d.stride(0), p2d.shape[0],
                                       p2d.shape[1], N.ptr(row_flags), float(lr), beta1, beta2, eps, wd, bc1, bc2s,
                                       N.ptr(hyper_dev), N.ptr(clip), int(clear_grad), N.stream()), "adam_table")


def clip_coef(acc64, max_norm: float, coef, norm_out=None) -> None:
    N.check(N.lib().b200rec_clip_coef(N.ptr(acc64), max_norm, N.ptr(coef), N.ptr(norm_out), N.stream()), "clip_coef")


def adam_dense_(p, g, m, v, lr, beta1, beta2, eps, wd, step: int, clip=None, clear_grad: bool = False) -> None:
    bc1 = 1.0 - beta1 ** step
    bc2s = (1.0 - beta2 ** step) ** 0.5
    N.check(N.lib().b200rec_adam_dense(N.ptr(p), N.ptr(g), N.ptr(m), N.ptr(v), p.numel(), lr, beta1, beta2, eps, wd, bc1,
                                       bc2s, N.ptr(clip), int(clear_grad), N.stream()), "adam_dense")


def sparse_adam_(table, m, v, rows, grads, n, lr, beta1, beta2, eps, step: int, clip=None) -> None:
    bc1 = 1.0 - beta1 ** step
    bc2s = (1.0 - beta2 ** step) ** 0.5
    N.check(N.lib().b200rec_sparse_adam(N.ptr(table), N.ptr(m), N.ptr(v), table.stride(0), grads.shape[1], N.ptr(rows),
                                        N.ptr(grads), N.ptr(n), rows.shape[0], lr, beta1, beta2, eps, bc1, bc2s,
                                        N.ptr(clip), N.stream()), "sparse_adam")


def train_step_begin(step_dev, lr_dev, beta1: float, beta2: float, hyper_dev, salt_key: int) -> None:
    N.check(N.lib().b200rec_train_step_begin(N.ptr(step_dev), N.ptr(lr_dev), beta1, beta2, N.ptr(hyper_dev),
                                             salt_key & 0xFFFFFFFFFFFFFFFF, N.stream()), "train_step_begin")


def adam_dense_dev_(p, g, m, v, beta1, beta2, eps, wd, hyper_dev, clip=None, clear_grad: bool = False) -> None:
    N.check(N.lib().b200rec_adam_dense_dev(N.ptr(p), N.ptr(g), N.ptr(m), N.ptr(v), p.numel(), beta1, beta2, eps, wd,
                                           N.ptr(hyper_dev), N.ptr(clip), int(clear_grad), N.stream()), "adam_dense_dev")


def sparse_adam_dev_(table, m, v, rows, grads, n, beta1, beta2, eps, hyper_dev, clip=None) -> None:
    N.check(N.lib().b200rec_sparse_adam_dev(N.ptr(table), N.ptr(m), N.ptr(v), table.stride(0), grads.shape[1],
                                            N.ptr(rows), N.ptr(grads), N.ptr(n), rows.shape[0], beta1, beta2, eps,
                                            N.ptr(hyper_dev), N.ptr(clip), N.stream()), "sparse_adam_dev")


# ------------------------------------------------------------------------------------------------ device-side batch feed
def gather_rows(table: torch.Tensor, idx: torch.Tensor, err: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out[b, :] = table[idx[b], :] (fp32 feature rows); an out-of-range index raises err (int32[1]) to 1."""
    assert table.dtype == torch.float32 and table.dim() == 2 and table.stride(1) == 1 and idx.dtype == torch.int64
    B, width = idx.numel(), table.shape[1]
    if out is None:
        out = torch.empty((B, width), dtype=torch.float32, device=table.device)
    N.check(N.lib().b200rec_gather_rows(N.ptr(table), table.shape[0], width, table.stride(0), N.ptr(idx), B, N.ptr(out),
                                        out.stride(0), N.ptr(err), N.stream()), "gather_rows")
    return out


def sample_negatives(user_of_row: torch.Tensor, pos_indptr: torch.Tensor, pos_items: torch.Tensor, num_items: int,
                     num_negatives: int, seed: int, row_base: int, err: torch.Tensor) -> torch.Tensor:
    """[B, num_negatives] int64: distinct items, uniform over the items each row's user has not interacted with."""
    B = user_of_row.numel()
    out = torch.empty((B, num_negatives), dtype=torch.int64, device=user_of_row.device)
    N.check(N.lib().b200rec_sample_negatives(N.ptr(user_of_row), B, N.ptr(pos_indptr), N.ptr(pos_items),
                                             pos_indptr.numel() - 1, num_items, num_negatives,
                                             seed & 0xFFFFFFFFFFFFFFFF, row_base, N.ptr(out), N.ptr(err), N.stream()),
            "sample_negatives")
    return out
