"""Drop-in B200 mirror of the exact inner-product path of the reference's `src/serving/retrieval.py`:
IndexBase (:16-46), FaissIndex Flat/cosine branch (:49-329) and RetrievalEngine (:505-692).

`B200FlatIndex.index` is a `FlatIPDeviceIndex`, the faiss-shaped object: `add(x)`, `search(q, k) -> (D, I)` with
faiss.IndexFlatIP's array contract (fp32 scores descending, int64 labels, -1 / -FLT_MAX padding).  The catalogue lives
in HBM as a bf16 tensor-core operand; scoring + top-K run in one fused tcgen05 kernel (csrc/topk.cu).  IVF / L2 /
Annoy / Milvus are outside this hot path (SURVEY.md section 8) and are rejected loudly.
"""
from __future__ import annotations

import logging
import pickle
import struct
import heapq
import time
import weakref
from abc import ABC, abstractmethod
from pathlib import Path
from typing import Any, Dict, List, Optional, Tuple

import numpy as np
import torch

from . import kernels as K
from ._native import pad64

logger = logging.getLogger("b200rec")
FLT_MAX = float(np.finfo(np.float32).max)


def _max_dimension(storage: str) -> int:
    """Largest row dimension the top-K kernels have a plan for: the resident query tile holds ld = terms * pad64(d)
    bf16 columns (terms = 3 for fp32 storage), which the library answers without a GPU."""
    terms = 1 if storage == "bf16" else 3
    d = 0
    while K.topk_workspace_bytes(1, terms * (d + 64), 1, 1) > 0:
        d += 64
    return d


def check_dimension(d: int, storage: str) -> None:
    """ValueError when d-dimensional rows in this storage cannot be searched, before any row reaches the device."""
    if d < 1:
        raise ValueError(f"dimension must be >= 1 (got {d})")
    if K.topk_workspace_bytes(1, (1 if storage == "bf16" else 3) * pad64(d), 1, 1) > 0:
        return
    msg = f"dimension {d} is too large: the largest supported d is {_max_dimension(storage)} for storage={storage!r}"
    if storage != "bf16":
        msg += f"; storage='bf16' lifts the limit to {_max_dimension('bf16')}"
    raise ValueError(msg)


def check_rows(rows, ntotal: int, what: str) -> np.ndarray:
    """Host validation of a row list (before anything reaches the device): 1-D integers in [0, ntotal), as int64."""
    r = np.asarray(rows.detach().cpu() if torch.is_tensor(rows) else rows)
    if r.ndim != 1:
        raise ValueError(f"{what}: rows must be a 1-D integer array (got shape {r.shape})")
    if r.size == 0:
        return np.zeros(0, dtype=np.int64)
    if not np.issubdtype(r.dtype, np.integer):
        raise ValueError(f"{what}: rows must be an integer array (got {r.dtype})")
    r = r.astype(np.int64, copy=False)
    bad = (r < 0) | (r >= ntotal)
    if bad.any():
        raise ValueError(f"{what}: row {int(r[bad][0])} is outside [0, ntotal = {ntotal})")
    return r


class IndexBase(ABC):
    """Abstract base class for ANN indices (reference retrieval.py:16-46)."""

    @abstractmethod
    def build(self, embeddings: np.ndarray, ids: List[str]):
        pass

    @abstractmethod
    def search(self, query_embeddings: np.ndarray, k: int = 10) -> Tuple[List[List[str]], List[List[float]]]:
        pass

    @abstractmethod
    def add(self, embeddings: np.ndarray, ids: List[str]):
        pass

    @abstractmethod
    def save(self, path: str):
        pass

    @abstractmethod
    def load(self, path: str):
        pass


class RowFilter:
    """A fixed set of LOCAL rows of one `FlatIPDeviceIndex` (faiss' IDSelectorBatch semantics): built by
    `FlatIPDeviceIndex.row_filter`, passed as `sel=` to `search_device` / `search`, which then return the exact top-k
    over these rows only.  Rows added to the index after the filter was built are not allowed.

    `rows` (int64, ascending, on the device) and `bits` (the IDSelectorBitmap of those rows, int32 words) are built once.
    `compacted()` is the catalogue operand restricted to the allowed rows ([n_allowed, ld] bf16, n_allowed * ld * 2
    bytes: 2.56 GB for an all-allowed filter over 10 M x 128 rows), gathered on first use and kept with the filter, so a
    filter reused across requests ("in stock") pays the gather once; flat-index rows never move, so `add` does not
    invalidate it.

    On a mutated index the filter keeps its row set and answers over (filter rows AND live rows) with the current row
    contents: `update_rows` / `remove_rows` patch the compacted copy in place (and its live bitmap in compact-row space,
    `_compact_bits`), the bitmap path ANDs `bits` with the index's live bits once per mutation epoch.  `compact()`
    renumbers the rows, after which the filter is rejected (ValueError)."""

    def __init__(self, index: "FlatIPDeviceIndex", rows: np.ndarray):
        self.index = index
        self.n_bits = index.ntotal
        self.n_allowed = int(rows.size)
        self.generation = index._generation
        self.rows = torch.from_numpy(np.ascontiguousarray(rows, dtype=np.int64)).to(index.device)
        self.bits = K.rows_to_bitmap(self.rows, max(self.n_bits, 1))
        self._compact: Optional[torch.Tensor] = None
        self._compact_bits: Optional[torch.Tensor] = None     # compact-row live bits, once the index has removed rows
        self._live_and: Optional[Tuple[int, torch.Tensor]] = None   # (mutation epoch, bits AND live bits)

    @property
    def fraction(self) -> float:
        """Allowed share of the rows the index held when the filter was built."""
        return self.n_allowed / max(self.n_bits, 1)

    def compacted(self) -> torch.Tensor:
        if self._compact is None:
            ix = self.index
            out = torch.empty((self.n_allowed, ix.ld), dtype=torch.bfloat16, device=ix.device)
            err = torch.zeros((1,), dtype=torch.int32, device=ix.device)
            # bf16 rows viewed as fp32 words (ld * 2 bytes is a multiple of 128 B): the feed's row gather does the copy
            K.gather_rows(ix._cat[: self.n_bits].view(torch.float32), self.rows, err, out=out.view(torch.float32))
            self._compact = out
            if ix._n_dead > 0:                   # rows of the filter removed before the gather stay in, bit cleared
                r = self.rows                    # compact bit j = live bit of row rows[j], packed on the device
                bit = (ix._live_bits[r >> 5] >> (r & 31)) & 1
                b = torch.nn.functional.pad(bit, (0, (-self.n_allowed) % 32)).view(-1, 32)
                words = (b << torch.arange(32, device=ix.device)).sum(1)
                self._compact_bits = torch.where(words >= 1 << 31, words - (1 << 32), words).to(torch.int32)
            ix._compact_filters.add(self)        # patched by every later mutation of the index
        return self._compact

    def live_bits(self) -> torch.Tensor:
        """`bits` AND the index's live-row bits (bitmap path on an index with removed rows), cached per mutation epoch."""
        ix = self.index
        if self._live_and is None or self._live_and[0] != ix._epoch:
            self._live_and = (ix._epoch, torch.bitwise_and(self.bits, ix._live_bits[: self.bits.numel()]))
        return self._live_and[1]


class FlatIPDeviceIndex:
    """faiss.IndexFlatIP on one B200: rows appended with `add`, exact `search`.

    storage "bf16": rows rounded to bf16 (BASELINE config 3; scores are exact fp32 sums of the rounded products).
    storage "fp32": for the reference-scale catalogues where scores and ids must be those of a CPU fp32 search.  Rows
    are kept twice: as fp32 and as split-bf16 x3 tensor-core operands.  The fused pass selects k + RESCORE_MARGIN
    candidates with 3 piece products (|err| <= ~1e-5 * |q||x|), `b200rec_rescore_fp32` recomputes those candidates'
    inner products with fp32 FMAs from the fp32 rows and a final select orders them (score desc, row asc): scores are
    fp32-exact (~1e-7), ids differ from an fp32 CPU search only where fp32 summation order itself decides.

    Mutable catalogue: `update_rows(rows, x)` overwrites row slots in place, `remove_rows(rows)` tombstones them and
    `compact()` drops the removed slots (the only operation that renumbers rows).  `ntotal` counts row slots, `n_live`
    the rows a search can return; every search path returns live rows only.  Until the first removal the index runs
    exactly the unmutated code; after it, a live-row bitmap (one bit per slot, kept on the device and mirrored on the
    host) is tested inside the fused kernel.  Mutations are enqueued on the caller's current CUDA stream: a search issued
    on that stream after a mutation call has returned sees the mutation (`search` / `search_stream` search on the current
    stream, so batches submitted after an update see it).  The older row-shard steps (`sample_device`, `sample_fanout`,
    `search_fanout`, `sample_filtered`, `search_filtered_shard`) do not read the live bitmap and refuse an index with
    removed rows; `sample_shard` / `search_shard`, which `dist.ShardedFlatIndex` runs, read it.
    """

    @staticmethod
    def rescore_margin(k: int) -> int:
        """Extra candidates the tensor-core pass hands to the exact fp32 re-scoring: enough that the true top-k are
        inside unless more than this many rows lie within the 3-product error of the k-th score."""
        return max(16, k // 4)

    # Filtered search over a compacted copy of the allowed rows below this allowed fraction, with the row bitmap tested
    # inside the fused kernel above it.  Measured on config 3 (DESIGN.md section 4, tools/filtered_search.py): the
    # cached compact search is faster at every fraction, and at f <= 0.5 by 1.6-44x; at f = 1 it gains 8-13 % for a
    # second 2.56 GB copy of the catalogue and a 1.8-2.0 ms first gather, so near-complete filters keep the bitmap.
    FILTER_COMPACT_BELOW = 0.75

    def __init__(self, d: int, storage: str = "fp32", device: Optional[torch.device] = None, row_offset: int = 0):
        if storage not in ("bf16", "fp32"):
            raise ValueError("storage must be 'bf16' or 'fp32'")
        check_dimension(int(d), storage)
        if not torch.cuda.is_available():
            raise RuntimeError("FlatIPDeviceIndex needs a CUDA (sm_100a) device; there is no CPU search path")
        self.d = int(d)
        self.storage = storage
        self.terms = 1 if storage == "bf16" else 3
        self.kpad = pad64(self.d)
        self.ld = self.terms * self.kpad
        self.device = device or torch.device("cuda", torch.cuda.current_device())
        self.row_offset = int(row_offset)
        self.ntotal = 0
        self.is_trained = True
        self._cat = torch.empty((0, self.ld), dtype=torch.bfloat16, device=self.device)
        self._f32 = torch.empty((0, self.d), dtype=torch.float32, device=self.device) if storage == "fp32" else None
        self._ws: Optional[torch.Tensor] = None
        # mutation state: live bits allocated on the first removal (all ones over the reserved slots, so `add` never
        # touches them), host mirror of the same bits, removed-slot count, epoch (bumped by every mutation) and
        # generation (bumped by compact(): row filters of an older generation are rejected)
        self._live_bits: Optional[torch.Tensor] = None
        self._live_host: Optional[np.ndarray] = None
        self._n_dead = 0
        self._epoch = 0
        self._generation = 0
        self._compact_filters: "weakref.WeakSet[RowFilter]" = weakref.WeakSet()

    # ------------------------------------------------------------------ rows
    def _reserve(self, n: int) -> None:
        if n <= self._cat.shape[0]:
            return
        cap = max(n, int(self._cat.shape[0] * 1.5), 1024)
        new = torch.empty((cap, self.ld), dtype=torch.bfloat16, device=self.device)
        new[: self.ntotal] = self._cat[: self.ntotal]
        self._cat = new
        if self._f32 is not None:
            nf = torch.empty((cap, self.d), dtype=torch.float32, device=self.device)
            nf[: self.ntotal] = self._f32[: self.ntotal]
            self._f32 = nf
        if self._live_bits is not None:         # new slots are live
            nb = torch.full(((cap + 31) // 32,), -1, dtype=torch.int32, device=self.device)
            nb[: self._live_bits.numel()] = self._live_bits
            self._live_bits = nb
            nh = np.ones(cap, dtype=bool)
            nh[: self._live_host.size] = self._live_host
            self._live_host = nh

    def add(self, x, normalize: bool = False) -> None:
        """Append rows (np.ndarray or torch tensor [n, d], any float dtype).  normalize=True applies faiss.normalize_L2."""
        xt = torch.as_tensor(x)
        if xt.dim() != 2 or xt.shape[1] != self.d:
            raise ValueError(f"expected [n, {self.d}] rows, got {tuple(xt.shape)}")
        n = xt.shape[0]
        if n == 0:
            return
        self._reserve(self.ntotal + n)
        step = 1 << 20
        for s in range(0, n, step):
            chunk = xt[s:s + step].to(self.device, dtype=torch.float32, non_blocking=True).contiguous()
            m = chunk.shape[0]
            dst = self._cat[self.ntotal + s: self.ntotal + s + m]
            f32 = self._f32[self.ntotal + s: self.ntotal + s + m] if self._f32 is not None else None
            K.N.check(K.N.lib().b200rec_normalize_rows(K.N.ptr(chunk), m, self.d, chunk.stride(0), int(normalize), 1,
                                                       K.N.ptr(f32), self.d, None, K.N.ptr(dst), self.kpad, self.terms,
                                                       1, K.N.stream()), "normalize_rows")
        self.ntotal += n

    def add_bf16_rows(self, rows: torch.Tensor) -> None:
        """Append rows that already are bf16 operands [n, ld] on the device (bulk loaders; storage 'bf16' only).  Into an
        empty index a contiguous tensor is taken over without a copy: the index then owns it, and `update_rows` writes
        into that tensor (until a later `add` or `compact()` moves the rows to storage of the index's own)."""
        assert self.storage == "bf16" and rows.dtype == torch.bfloat16 and rows.shape[1] == self.ld
        if self.ntotal == 0 and rows.is_contiguous() and rows.device == self.device:
            self._cat = rows
        else:
            self._reserve(self.ntotal + rows.shape[0])
            self._cat[self.ntotal: self.ntotal + rows.shape[0]] = rows
        self.ntotal += rows.shape[0]

    # ------------------------------------------------------------------ mutation
    @property
    def n_live(self) -> int:
        """Rows a search can return: ntotal minus the removed slots."""
        return self.ntotal - self._n_dead

    def _check_rows(self, rows, what: str) -> np.ndarray:
        return check_rows(rows, self.ntotal, what)

    def _ensure_live(self) -> None:
        if self._live_bits is None:
            cap = self._cat.shape[0]
            self._live_bits = torch.full(((cap + 31) // 32,), -1, dtype=torch.int32, device=self.device)
            self._live_host = np.ones(cap, dtype=bool)

    def _patch_filters(self, rows_dev: torch.Tensor, update: bool) -> None:
        """One patch launch per cached compacted filter: copy updated rows in / set or clear their compact live bits."""
        for f in list(self._compact_filters):
            if f._compact is None or f.n_allowed == 0 or f.generation != self._generation:
                continue
            if update:
                K.patch_compacted(rows_dev, f.rows, self._cat, f._compact, f._compact_bits, True)
            else:
                if f._compact_bits is None:
                    f._compact_bits = torch.full(((f.n_allowed + 31) // 32,), -1, dtype=torch.int32, device=self.device)
                K.patch_compacted(rows_dev, f.rows, None, None, f._compact_bits, False)

    def update_rows(self, rows, x, normalize: bool = False) -> None:
        """Overwrite row slots in place: x[i] (np.ndarray or torch tensor [n, d], any float dtype) goes to slot rows[i]
        (the bf16 operand and, for storage 'fp32', the fp32 rows); normalize=True applies faiss.normalize_L2 as `add`
        does.  A removed slot is revived.  Duplicate rows: the last occurrence wins.  ValueError (before any device
        work) for rows outside [0, ntotal), non-integer rows or a shape mismatch."""
        r = self._check_rows(rows, "update_rows")
        xt = torch.as_tensor(x)
        if xt.dim() != 2 or xt.shape[1] != self.d or xt.shape[0] != r.size:
            raise ValueError(f"update_rows: expected [{r.size}, {self.d}] rows, got {tuple(xt.shape)}")
        if r.size == 0:
            return
        u, first_rev = np.unique(r[::-1], return_index=True)     # ascending distinct rows, last occurrence of each
        pos = r.size - 1 - first_rev
        if not np.array_equal(pos, np.arange(r.size)):
            xt = xt[torch.from_numpy(pos).to(xt.device)]
        rows_dev = torch.from_numpy(u).to(self.device, non_blocking=True)
        n, step = u.size, 1 << 20
        for s in range(0, n, step):
            chunk = xt[s:s + step].to(self.device, dtype=torch.float32, non_blocking=True).contiguous()
            K.update_rows(chunk, rows_dev[s:s + chunk.shape[0]], self._cat, self.kpad, self.terms, self._f32,
                          self._live_bits, normalize)
        if self._live_host is not None:
            self._n_dead -= int(np.count_nonzero(~self._live_host[u]))
            self._live_host[u] = True
        self._epoch += 1
        self._patch_filters(rows_dev, update=True)

    def remove_rows(self, rows) -> int:
        """Tombstone row slots (they stay in place until `compact()`); returns how many of them were live.  Removed
        and duplicate rows are harmless; ValueError for rows outside [0, ntotal) or non-integer rows."""
        u = np.unique(self._check_rows(rows, "remove_rows"))
        if u.size == 0:
            return 0
        self._ensure_live()
        gone = u[self._live_host[u]]
        if gone.size == 0:
            return 0
        self._live_host[gone] = False
        self._n_dead += int(gone.size)
        self._epoch += 1
        rows_dev = torch.from_numpy(gone).to(self.device, non_blocking=True)
        K.clear_row_bits(rows_dev, self._live_bits, self.ntotal)
        self._patch_filters(rows_dev, update=False)
        return int(gone.size)

    def compact(self) -> np.ndarray:
        """Drop the removed slots (the live rows keep their order): returns the old -> new row map (int64 [old ntotal],
        -1 for removed rows).  Every RowFilter built before is rejected afterwards."""
        n = self.ntotal
        keep = np.flatnonzero(self._live_host[:n]) if self._live_host is not None else np.arange(n, dtype=np.int64)
        remap = np.full(n, -1, dtype=np.int64)
        remap[keep] = np.arange(keep.size, dtype=np.int64)
        if keep.size < n:
            idx = torch.from_numpy(keep).to(self.device)
            err = torch.zeros((1,), dtype=torch.int32, device=self.device)
            new = torch.empty((keep.size, self.ld), dtype=torch.bfloat16, device=self.device)
            nf = torch.empty((keep.size, self.d), dtype=torch.float32, device=self.device) if self._f32 is not None else None
            if keep.size:
                K.gather_rows(self._cat[:n].view(torch.float32), idx, err, out=new.view(torch.float32))
                if nf is not None:
                    K.gather_rows(self._f32[:n], idx, err, out=nf)
            self._cat, self._f32 = new, nf
            self.ntotal = int(keep.size)
        self._live_bits, self._live_host, self._n_dead = None, None, 0
        self._epoch += 1
        self._generation += 1
        self._compact_filters = weakref.WeakSet()
        return remap

    def _require_all_live(self, what: str) -> None:
        if self._n_dead:
            raise ValueError(f"{what}: the index has {self._n_dead} removed rows and row-sharded search does not read "
                             "the live-row bitmap; compact() it first")

    def _check_filter(self, sel: RowFilter) -> None:
        if sel.index is not self:
            raise ValueError("the row filter was built for another index")
        if sel.generation != self._generation:
            raise ValueError("the row filter was built before compact() renumbered the rows; build it again")

    def reconstruct_n(self, i0: int = 0, n: Optional[int] = None) -> np.ndarray:
        n = self.ntotal - i0 if n is None else n
        if self._f32 is not None:
            return self._f32[i0:i0 + n].cpu().numpy()
        return self._cat[i0:i0 + n, : self.d].float().cpu().numpy()

    # ------------------------------------------------------------------ search
    def prepare_queries(self, q, normalize: bool = False) -> torch.Tensor:
        qt = torch.as_tensor(q)
        if qt.dim() == 1:
            qt = qt.reshape(1, -1)
        if qt.shape[1] != self.d:
            raise ValueError(f"expected [nq, {self.d}] queries, got {tuple(qt.shape)}")
        qt = qt.to(self.device, dtype=torch.float32, non_blocking=True).contiguous()
        keep = self.storage == "fp32"
        y, _, qop = K.normalize_rows(qt, normalize=normalize, faiss_rule=True, want_f32=keep and normalize,
                                     want_norms=False, terms=self.terms, side=0)
        if keep:
            qop._b200_f32 = y if normalize else qt       # the fp32 queries travel with their operand (exact re-scoring)
        return qop

    def _workspace(self, nq: int, k: int, n: Optional[int] = None) -> torch.Tensor:
        need = K.topk_workspace_bytes(self.ntotal if n is None else n, self.ld, nq, k)
        if need == 0:
            raise RuntimeError(f"b200rec flat_ip_topk: {K.N.last_error()}")
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty((need,), dtype=torch.uint8, device=self.device)
        return self._ws

    def has_sample_pass(self, nq: int, k: int) -> bool:
        return self.ntotal > 0 and K.topk_has_sample(self.ntotal, self.ld, nq, k)

    def sample_device(self, q_op: torch.Tensor, k: int, k_out: Optional[int] = None, shards: int = 1) -> torch.Tensor:
        """Sampling pass only: the k_out largest group maxima per query [nq, k_out] (exchanged between row shards)."""
        self._require_all_live("sample_device")
        return K.topk_sample(self._cat[: self.ntotal], q_op, k, self._workspace(q_op.shape[0], k), k_out, shards)

    def sample_fanout(self, q_op: torch.Tensor, k: int, k_out: int, shards: int, dst_vals) -> None:
        """Sampling pass whose [nq, k_out] maxima are stored to every address in dst_vals (peer gather buffers)."""
        self._require_all_live("sample_fanout")
        K.topk_sample_fanout(self._cat[: self.ntotal], q_op, k, k_out, shards, dst_vals, self._workspace(q_op.shape[0], k))

    def search_fanout(self, q_op: torch.Tensor, k: int, tau_init, dst_scores, dst_ids) -> None:
        """Local top-k (global row ids) stored to every (dst_scores[d], dst_ids[d]) address (peer gather buffers)."""
        self._require_all_live("search_fanout")
        K.flat_ip_topk_fanout(self._cat[: self.ntotal], q_op, k, self.row_offset, tau_init, dst_scores, dst_ids,
                              self._workspace(q_op.shape[0], k))

    def row_filter(self, rows=None, mask=None) -> RowFilter:
        """Row filter over the rows held now: `rows` (int array, numpy or torch; out-of-range and duplicate rows are
        ignored) or `mask` (bool array of length <= ntotal; missing tail = not allowed)."""
        if (rows is None) == (mask is None):
            raise ValueError("row_filter takes exactly one of rows= or mask=")
        if mask is not None:
            m = np.asarray(mask.cpu() if torch.is_tensor(mask) else mask)
            if m.dtype != np.bool_ or m.ndim != 1 or m.size > self.ntotal:
                raise ValueError(f"mask must be a 1-D bool array of length <= ntotal ({self.ntotal})")
            r = np.flatnonzero(m)
        else:
            r = np.asarray(rows.cpu() if torch.is_tensor(rows) else rows).reshape(-1)
            if r.size and not np.issubdtype(r.dtype, np.integer):
                raise ValueError("rows must be an integer array")
            r = r.astype(np.int64, copy=False)
            r = np.unique(r[(r >= 0) & (r < self.ntotal)])
        return RowFilter(self, r)

    # ------------------------------------------------------------------ filtered row-shard steps (dist.ShardedFlatIndex)
    def _shard_operand(self, sel: RowFilter, compact: Optional[bool]):
        """(catalogue, allow_bits, allow_n, remap_rows) a filtered row-shard step runs over: the bitmap over the local
        catalogue, or the compacted allowed rows with their local row list (compact = None: chosen from the LOCAL
        allowed fraction, as search_device does).  No allowed row: (None, bits, 0, None), which the kernels answer with
        padding rows."""
        if self.storage != "bf16":
            raise ValueError("row-sharded filtered search needs bf16 storage (an fp32-storage shard re-scores its "
                             "candidates from fp32 rows, which the sharded exchange does not carry)")
        self._check_filter(sel)
        if sel.n_allowed == 0:
            return None, sel.bits, 0, None
        if compact is None:
            compact = sel.fraction < self.FILTER_COMPACT_BELOW
        if compact:
            return sel.compacted(), None, 0, sel.rows
        return self._cat[: self.ntotal], sel.bits, sel.n_bits, None

    def sample_filtered(self, q_op: torch.Tensor, k: int, k_out: int, shards: int, sel: RowFilter, dst=None,
                        compact: Optional[bool] = None) -> Optional[torch.Tensor]:
        """Sampling pass of a filtered row-sharded search: the k_out best group maxima per query over the allowed rows
        only, sampled for `shards` pooled shards; -FLT_MAX rows when this shard has no allowed row or no sampling pass
        for the shape.  Returned [nq, k_out], or stored to every address in `dst` (peer gather buffers)."""
        self._require_all_live("sample_filtered")
        cat, bits, allow_n, _ = self._shard_operand(sel, compact)
        ws = None if cat is None else self._workspace(q_op.shape[0], k, cat.shape[0])
        return K.topk_sample_filtered(cat, q_op, k, k_out, shards, bits, allow_n, ws, dst)

    def search_filtered_shard(self, q_op: torch.Tensor, k: int, sel: RowFilter, tau, out=None, dst=None,
                              compact: Optional[bool] = None):
        """Local exact top-k over the allowed rows from the pooled threshold `tau` ([nq] lower bounds of the GLOBAL k-th
        allowed score, or None), global row ids (row_offset added, compact ids mapped back inside the select kernel),
        -1 / -FLT_MAX padding.  Returns (D, I) (written into `out` when given), or stores the rows to every
        (dst[0][d], dst[1][d]) address and returns None."""
        self._require_all_live("search_filtered_shard")
        cat, bits, allow_n, remap = self._shard_operand(sel, compact)
        ws = None if cat is None else self._workspace(q_op.shape[0], k, cat.shape[0])
        if dst is not None:
            K.flat_ip_topk_filtered_fanout(cat, q_op, k, self.row_offset, bits, allow_n, remap, tau, dst[0], dst[1], ws)
            return None
        nq = q_op.shape[0]
        d, i = out if out is not None else (torch.empty((nq, k), dtype=torch.float32, device=self.device),
                                            torch.empty((nq, k), dtype=torch.int64, device=self.device))
        K.flat_ip_topk_filtered_fanout(cat, q_op, k, self.row_offset, bits, allow_n, remap, tau, [d.data_ptr()],
                                       [i.data_ptr()], ws)
        return d, i

    # ------------------------------------------------------------------ live-aware row-shard steps (dist.ShardedFlatIndex)
    def _live_operand(self, sel: Optional[RowFilter]):
        """(catalogue, allow_bits, allow_n, remap_rows) a row-shard step runs over on an index with removed rows: the
        live bits over the local catalogue, a bitmap filter ANDed with them, or a compacted filter's rows with its
        compact-row live bits and its local row list.  No live row: (None, None, 0, None), answered with padding."""
        if self.storage != "bf16":
            raise ValueError("row-sharded search over an index with removed rows needs bf16 storage (an fp32-storage "
                             "shard re-scores its candidates from fp32 rows, which the sharded exchange does not carry)")
        if sel is None:
            if self.n_live == 0:
                return None, None, 0, None
            return self._cat[: self.ntotal], self._live_bits, self.ntotal, None
        cat, bits, allow_n, remap = self._shard_operand(sel, None)
        if cat is None:
            return None, None, 0, None
        if remap is None:
            return cat, sel.live_bits(), allow_n, None
        return cat, sel._compact_bits, sel.n_allowed, remap

    def sample_shard(self, q_op: torch.Tensor, k: int, k_out: Optional[int] = None, shards: int = 1,
                     sel: Optional[RowFilter] = None, dst=None) -> Optional[torch.Tensor]:
        """Sampling step of a row-sharded search over the live (and, with `sel`, allowed) rows: the k_out (default k)
        best group maxima per query [nq, k_out], or stored to every address in `dst`.  An index with no removed row runs
        exactly sample_device / sample_fanout / sample_filtered (unfiltered: None when the shape has no sampling pass);
        one with removed rows runs the masked sampling pass and always answers, with -FLT_MAX rows where it has nothing
        to sample, so a shard's removals never change what the other shards do."""
        k_out = k if k_out is None else k_out
        if self._n_dead == 0:
            if sel is not None:
                return self.sample_filtered(q_op, k, k_out, shards, sel, dst=dst)
            if dst is not None:
                self.sample_fanout(q_op, k, k_out, shards, dst)
                return None
            if not self.has_sample_pass(q_op.shape[0], k):
                return None
            return self.sample_device(q_op, k, k_out, shards)
        cat, bits, allow_n, _ = self._live_operand(sel)
        ws = None if cat is None else self._workspace(q_op.shape[0], k, cat.shape[0])
        return K.topk_sample_filtered(cat, q_op, k, k_out, shards, bits, allow_n, ws, dst)

    def search_shard(self, q_op: torch.Tensor, k: int, tau, sel: Optional[RowFilter] = None, out=None, dst=None):
        """Local exact top-k of a row-sharded search over the live (and, with `sel`, allowed) rows from the pooled
        threshold `tau` ([nq] or None), global row ids, -1 / -FLT_MAX padding.  Returns (D, I) (written into `out` when
        given), or stores the rows to every (dst[0][d], dst[1][d]) address and returns None.  An index with no removed
        row runs exactly search_device(tau_init=) / search_fanout / search_filtered_shard; one with removed rows runs one
        fused search that tests the live bits (and the filter) and maps compacted ids back, bf16 storage only."""
        if self._n_dead == 0:
            if sel is not None:
                return self.search_filtered_shard(q_op, k, sel, tau, out=out, dst=dst)
            if dst is not None:
                self.search_fanout(q_op, k, tau, dst[0], dst[1])
                return None
            return self.search_device(q_op, k, tau_init=tau, out=out)
        cat, bits, allow_n, remap = self._live_operand(sel)
        ws = None if cat is None else self._workspace(q_op.shape[0], k, cat.shape[0])
        if dst is not None:
            K.flat_ip_topk_masked_fanout(cat, q_op, k, self.row_offset, bits, allow_n, remap, tau, dst[0], dst[1], ws)
            return None
        nq = q_op.shape[0]
        d, i = out if out is not None else (torch.empty((nq, k), dtype=torch.float32, device=self.device),
                                            torch.empty((nq, k), dtype=torch.int64, device=self.device))
        K.flat_ip_topk_masked_fanout(cat, q_op, k, self.row_offset, bits, allow_n, remap, tau, [d.data_ptr()],
                                     [i.data_ptr()], ws)
        return d, i

    def search_device(self, q_op: torch.Tensor, k: int, exclude_indptr=None, exclude_rows=None, tau_init=None,
                      out=None, sel: Optional[RowFilter] = None):
        """q_op: bf16 operand [nq, ld] on the device -> (D, I) device tensors (written into `out` when given).
        `sel` (a RowFilter of this index): exact top-k over the allowed rows only, -1 / -FLT_MAX padding past them."""
        nq = q_op.shape[0]
        if sel is not None:
            if exclude_indptr is not None or exclude_rows is not None:
                raise ValueError("a row filter cannot be combined with per-query exclusion lists")
            if tau_init is not None:
                raise ValueError("a row filter cannot be combined with tau_init (row-sharded search)")
            self._check_filter(sel)
            d, i = self._search_filtered(q_op, k, sel, sel.fraction < self.FILTER_COMPACT_BELOW)
            if out is not None:
                out[0].copy_(d)
                out[1].copy_(i)
                return out
            return d, i
        if self.ntotal == 0 or self._n_dead == self.ntotal:
            if out is not None:
                out[0].fill_(-FLT_MAX)
                out[1].fill_(-1)
                return out
            return (torch.full((nq, k), -FLT_MAX, dtype=torch.float32, device=self.device),
                    torch.full((nq, k), -1, dtype=torch.int64, device=self.device))
        q32 = getattr(q_op, "_b200_f32", None) if self._f32 is not None else None
        if self._n_dead > 0:                     # removed rows: the live bitmap as an allow bitmap, one path
            kk = k if q32 is None else min(k + self.rescore_margin(k), max(k, min(self.ntotal, 2048)))
            d, i = K.flat_ip_topk_masked(self._cat[: self.ntotal], q_op, kk, self.row_offset, exclude_indptr,
                                         exclude_rows, self._live_bits, self.ntotal, None,
                                         tau_init if q32 is None else None, self._workspace(nq, kk))
            if q32 is not None:
                exact = K.rescore_fp32(q32, self._f32[: self.ntotal], i, self.row_offset)
                d, i = K.topk_merge(exact.unsqueeze(0), i.unsqueeze(0), k)
            if out is not None:
                out[0].copy_(d)
                out[1].copy_(i)
                return out
            return d, i
        if q32 is None:
            return K.flat_ip_topk(self._cat[: self.ntotal], q_op, k, self.row_offset, exclude_indptr, exclude_rows,
                                  self._workspace(nq, k), tau_init, out)
        k_in = min(k + self.rescore_margin(k), max(k, min(self.ntotal, 2048)))
        _, cand = K.flat_ip_topk(self._cat[: self.ntotal], q_op, k_in, self.row_offset, exclude_indptr, exclude_rows,
                                 self._workspace(nq, k_in), None)   # tau_init bounds the k-th score, not the k_in-th
        exact = K.rescore_fp32(q32, self._f32[: self.ntotal], cand, self.row_offset)
        d, i = K.topk_merge(exact.unsqueeze(0), cand.unsqueeze(0), k)
        if out is not None:
            out[0].copy_(d)
            out[1].copy_(i)
            return out
        return d, i

    def _search_filtered(self, q_op: torch.Tensor, k: int, sel: RowFilter, compact: bool):
        """Both exact filtered paths: compact = search the gathered allowed rows and map the ids back through the row
        list; else the full catalogue with the row bitmap tested inside the fused kernel.  fp32 storage: k + margin
        candidates among the allowed rows, re-scored from the fp32 rows as in search_device."""
        nq = q_op.shape[0]
        q32 = getattr(q_op, "_b200_f32", None) if self._f32 is not None else None
        if compact and sel.n_allowed == 0:
            return (torch.full((nq, k), -FLT_MAX, dtype=torch.float32, device=self.device),
                    torch.full((nq, k), -1, dtype=torch.int64, device=self.device))
        kk = k if q32 is None else min(k + self.rescore_margin(k), max(k, min(self.ntotal, 2048)))
        if compact:
            cat = sel.compacted()
            if self._n_dead > 0 and sel._compact_bits is not None:   # compact live bits + remap in the same search
                d, i = K.flat_ip_topk_masked(cat, q_op, kk, self.row_offset, allow_bits=sel._compact_bits,
                                             allow_n=sel.n_allowed, remap_rows=sel.rows,
                                             workspace=self._workspace(nq, kk, cat.shape[0]))
            else:
                d, i = K.flat_ip_topk(cat, q_op, kk, 0, workspace=self._workspace(nq, kk, cat.shape[0]))
                K.remap_ids(i, sel.rows, self.row_offset)
        else:
            bits = sel.live_bits() if self._n_dead > 0 else sel.bits
            d, i = K.flat_ip_topk_filtered(self._cat[: self.ntotal], q_op, kk, bits, sel.n_bits, self.row_offset,
                                           self._workspace(nq, kk))
        if q32 is None:
            return d, i
        exact = K.rescore_fp32(q32, self._f32[: self.ntotal], i, self.row_offset)
        return K.topk_merge(exact.unsqueeze(0), i.unsqueeze(0), k)

    def search(self, q, k: int, normalize: bool = False, sel: Optional[RowFilter] = None) -> Tuple[np.ndarray, np.ndarray]:
        """faiss contract: (D float32 [nq,k] descending, I int64 [nq,k]) as numpy arrays — `index.search(q, k)` of
        reference retrieval.py:171.  Host queries travel through pinned staging buffers kept by the index; a filtered
        search (`sel`, see search_device) takes the blocking path."""
        if sel is not None or (torch.is_tensor(q) and q.is_cuda):
            d, i = self.search_device(self.prepare_queries(q, normalize), k, sel=sel)
            return d.cpu().numpy(), i.cpu().numpy()
        for out in self.search_stream([q], k, normalize):
            return out

    def search_stream(self, batches, k: int, normalize: bool = False, device_search=None):
        """Throughput form of `search` for a stream of HOST query batches (numpy [nq, d], any float dtype): yields one
        faiss-shaped (D, I) numpy pair per batch, in order.  Batch i+1's staging + host->device copy and batch i-1's
        device->host copy run on side streams while batch i is being searched, so a step costs max(search, copies)
        instead of their sum.  `device_search(q_op, k) -> (D, I)` device tensors (default: this index; row-sharded
        search passes its own)."""
        if device_search is None:                # pinned staging buffers are allocated once per (k, normalize)
            pipes = self.__dict__.setdefault("_pipes", {})
            pipe = pipes.get((k, normalize))
            if pipe is None:
                pipe = pipes[(k, normalize)] = HostPipeline(self, k, normalize, lambda q_op, kk: self.search_device(q_op, kk))
        else:
            pipe = device_search if isinstance(device_search, HostPipeline) else HostPipeline(self, k, normalize, device_search)
        pending = None
        for q in batches:
            ticket = pipe.submit(q)
            if pending is not None:
                yield pipe.collect(pending)
            pending = ticket
        if pending is not None:
            yield pipe.collect(pending)


class HostPipeline:
    """Double-buffered host <-> device path of `FlatIPDeviceIndex.search_stream`: two pinned query buffers, two pinned
    result buffers, one copy-in and one copy-out stream next to the caller's compute stream, CUDA events in between.
    `rows` (optional slice) limits the device->host copy to a sub-range of the queries (a row-sharded deployment
    returns each replica's share of the answers)."""

    DEPTH = 2

    def __init__(self, index: FlatIPDeviceIndex, k: int, normalize: bool, device_search, rows: Optional[slice] = None):
        self.index, self.k, self.normalize, self.device_search, self.rows = index, int(k), normalize, device_search, rows
        self.s_in = torch.cuda.Stream(device=index.device)
        self.s_out = torch.cuda.Stream(device=index.device)
        self.slots: List[Dict[str, Any]] = [dict() for _ in range(self.DEPTH)]
        self.n = 0
        self.h2d_bytes = 0
        self.d2h_bytes = 0

    def _slot(self, nq: int) -> Dict[str, Any]:
        sl = self.slots[self.n % self.DEPTH]
        if sl.get("nq") != nq:
            d, k, dev = self.index.d, self.k, self.index.device
            lo, hi = (0, nq) if self.rows is None else self.rows.indices(nq)[:2]
            sl.update(nq=nq, lo=lo, hi=hi,
                      q_host=torch.empty((nq, d), dtype=torch.float32).pin_memory(),
                      q_dev=torch.empty((nq, d), dtype=torch.float32, device=dev),
                      d_host=torch.empty((hi - lo, k), dtype=torch.float32).pin_memory(),
                      i_host=torch.empty((hi - lo, k), dtype=torch.int64).pin_memory(),
                      done=torch.cuda.Event(), copied=None, keep=None)
        return sl

    def submit(self, q) -> Dict[str, Any]:
        qn = np.asarray(q)
        if qn.ndim == 1:
            qn = qn.reshape(1, -1)
        if qn.shape[1] != self.index.d:
            raise ValueError(f"expected [nq, {self.index.d}] queries, got {tuple(qn.shape)}")
        sl = self._slot(qn.shape[0])
        if sl["copied"] is not None:
            sl["copied"].synchronize()          # the slot's previous results have left the device (and were collected)
        np.copyto(sl["q_host"].numpy(), qn, casting="same_kind")                  # staging (+ dtype cast) on the host
        cur = torch.cuda.current_stream(self.index.device)
        with torch.cuda.stream(self.s_in):
            sl["q_dev"].copy_(sl["q_host"], non_blocking=True)
            arrived = torch.cuda.Event()
            arrived.record(self.s_in)
        cur.wait_event(arrived)
        q_op = self.index.prepare_queries(sl["q_dev"], self.normalize)
        d, i = self.device_search(q_op, self.k)
        sl["done"].record(cur)
        sl["keep"] = (q_op, d, i)                # keep the device results alive until they are copied out
        with torch.cuda.stream(self.s_out):
            self.s_out.wait_event(sl["done"])
            sl["d_host"].copy_(d[sl["lo"]:sl["hi"]], non_blocking=True)
            sl["i_host"].copy_(i[sl["lo"]:sl["hi"]], non_blocking=True)
            copied = torch.cuda.Event()
            copied.record(self.s_out)
        sl["copied"] = copied
        self.n += 1
        self.h2d_bytes += qn.shape[0] * self.index.d * 4
        self.d2h_bytes += (sl["hi"] - sl["lo"]) * self.k * 12
        return sl

    def collect(self, sl: Dict[str, Any]) -> Tuple[np.ndarray, np.ndarray]:
        sl["copied"].synchronize()
        sl["keep"] = None
        return sl["d_host"].numpy().copy(), sl["i_host"].numpy().copy()   # the pinned buffers are reused two batches later


class B200FlatIndex(IndexBase):
    """`FaissIndex` on the exact Flat / inner-product branch (reference retrieval.py:49-329), B200-resident.

    config "updates": "warn" (default) keeps the reference's behaviour: `add` appends a row even for an id that is already
    indexed, `update` / `remove` only log the reference's warnings.  "in_place" makes the catalogue mutable: `add` and
    `update` are the same upsert (known ids are overwritten in place, new ids fill removed slots lowest first and then
    append, the last occurrence of a repeated id wins), `remove(ids)` tombstones the rows of known ids, and searches
    return live items only, so a streaming `RetrievalEngine.update_index` never returns an item twice.  `current_size`
    then counts live items, `id_map` / `reverse_id_map` hold live rows only, `save` writes the live rows renumbered
    densely and `compact()` drops removed slots."""

    def __init__(self, config: Optional[Dict[str, Any]] = None):
        self.config = config or {}
        self.dimension = self.config.get("dimension", 128)
        self.index_factory = self.config.get("index_factory", "Flat")
        self.metric = self.config.get("metric", "cosine")
        self.nprobe = self.config.get("nprobe", 20)
        self.use_gpu = True
        self.storage = self.config.get("storage", "fp32")
        check_dimension(int(self.dimension), self.storage)
        self.updates = self.config.get("updates", "warn")
        if self.updates not in ("warn", "in_place"):
            raise ValueError(f"updates {self.updates!r}: 'warn' (the reference: add appends, update / remove only warn) "
                             "or 'in_place' (upsert / remove on the live catalogue)")
        self.filter = self.config.get("filter", "post")
        if self.filter not in ("post", "exact"):
            raise ValueError(f"filter {self.filter!r}: 'post' (the reference's post-pass over the 2k best rows) or "
                             "'exact' (the exact top-k among the filter_ids rows)")
        if self.metric not in ("cosine", "ip", "inner_product"):
            raise ValueError(f"metric {self.metric!r}: only the cosine / inner-product path is B200-native "
                             "(IndexFlatL2 is outside the hot path)")
        self.index: Optional[FlatIPDeviceIndex] = None
        self.id_map: Dict[int, str] = {}
        self.reverse_id_map: Dict[str, int] = {}
        self.current_size = 0
        self._free: List[int] = []              # "in_place": removed slots, a min-heap (reused lowest first)

    def build(self, embeddings: np.ndarray, ids: List[str]):
        n_items = len(embeddings)
        logger.info("Building B200 flat index for %d items...", n_items)
        start = time.time()
        if "IVF" in self.index_factory and n_items >= 1024:
            logger.info("index_factory %r is approximate in the reference; the B200 index is always exact",
                        self.index_factory)
        self.index = FlatIPDeviceIndex(self.dimension, storage=self.storage)
        self.index.add(np.asarray(embeddings, dtype=np.float32), normalize=(self.metric == "cosine"))
        self.id_map = {}
        self.reverse_id_map = {}
        self._id_array = None
        for i, item_id in enumerate(ids):
            self.id_map[i] = item_id
            self.reverse_id_map[item_id] = i
        self.current_size = n_items
        self._free = []
        if self.updates == "in_place":           # a repeated id keeps its last row; the other rows are removed
            self._drop_unmapped_rows()
        logger.info("Index built in %.2f seconds", time.time() - start)

    def _n_rows(self) -> int:
        """Row slots the row -> id array spans: every row of the device index under "in_place", else current_size."""
        return self.index.ntotal if self.updates == "in_place" else self.current_size

    def _names(self) -> np.ndarray:
        """Row -> item id as one object array (the reference walks nq x k dict lookups in Python, retrieval.py:177-195)."""
        arr = getattr(self, "_id_array", None)
        n = self._n_rows()
        if arr is None or len(arr) != n:
            arr = np.empty(n, dtype=object)
            arr[:] = [self.id_map.get(i) for i in range(n)]
            self._id_array = arr
            self._mapped = np.fromiter((x is not None for x in arr), dtype=bool, count=n)
        return arr

    def _set_name(self, row: int, item_id: Optional[str]) -> None:
        """Keep the cached row -> id array in step with one in-place change (it is rebuilt when rows were appended)."""
        arr = getattr(self, "_id_array", None)
        if arr is not None and row < len(arr):
            arr[row] = item_id
            self._mapped[row] = item_id is not None

    def search(self, query_embeddings: np.ndarray, k: int = 10,
               filter_ids: Optional[List[str]] = None) -> Tuple[List[List[str]], List[List[float]]]:
        """FaissIndex.search (retrieval.py:141-197): exact top-k, rows mapped to item ids.  `filter_ids` under config
        "filter": "post" (default) is the reference's POST-filter over the k_search = min(2k, N) best rows (it may return
        fewer than k ids); under "exact" the result is the exact top-k among the rows of the known filter_ids
        (min(k, |allowed rows|) ids per query; unknown ids are ignored)."""
        if self.index is None:
            raise ValueError("Index not built yet")
        if not (torch.is_tensor(query_embeddings) and query_embeddings.is_cuda):   # device tensors skip the host round trip
            query_embeddings = np.asarray(query_embeddings).astype(np.float32)
        if len(query_embeddings.shape) == 1:
            query_embeddings = query_embeddings.reshape(1, -1)
        exact = filter_ids is not None and self.filter == "exact"
        if self.updates == "in_place" and self.current_size == 0:      # every item removed
            return [[] for _ in range(len(query_embeddings))], [[] for _ in range(len(query_embeddings))]
        if exact:
            rows = np.fromiter((self.reverse_id_map[x] for x in set(filter_ids) if x in self.reverse_id_map), np.int64)
            distances, indices = self.index.search(query_embeddings, k, normalize=(self.metric == "cosine"),
                                                   sel=self.index.row_filter(rows=rows))
        else:
            k_search = min(k * 2, self.current_size) if filter_ids else k
            distances, indices = self.index.search(query_embeddings, k_search, normalize=(self.metric == "cosine"))
        if self.current_size == 0:
            return [[] for _ in range(len(indices))], [[] for _ in range(len(indices))]
        names = self._names()
        keep = (indices >= 0) & (indices < self._n_rows())
        safe = np.where(keep, indices, 0)
        keep &= self._mapped[safe]
        picked = names[safe]
        if filter_ids is not None and not exact:                               # [] filters everything out, as the reference
            member = set(filter_ids).__contains__                              # one C-level pass over the candidates
            keep &= np.frompyfunc(member, 1, 1)(picked).astype(bool)
        if keep.all():
            return picked[:, :k].tolist(), distances[:, :k].astype(float).tolist()
        rank = np.cumsum(keep, axis=1)
        keep &= rank <= k                                                      # first k survivors of every row
        return ([picked[r][keep[r]].tolist() for r in range(len(indices))],
                [distances[r][keep[r]].astype(float).tolist() for r in range(len(indices))])

    def add(self, embeddings: np.ndarray, ids: List[str]):
        if self.index is None:
            raise ValueError("Index not built yet")
        if self.updates == "in_place":
            self._upsert(embeddings, ids)
            return
        embeddings = np.asarray(embeddings).astype(np.float32)
        self.index.add(embeddings, normalize=(self.metric == "cosine"))
        for i, item_id in enumerate(ids):
            new_idx = self.current_size + i
            self.id_map[new_idx] = item_id
            self.reverse_id_map[item_id] = new_idx
        self.current_size += len(embeddings)
        logger.info("Added %d items to index. Total size: %d", len(embeddings), self.current_size)

    def update(self, embeddings: np.ndarray, ids: List[str]):
        if self.updates == "in_place":
            if self.index is None:
                raise ValueError("Index not built yet")
            self._upsert(embeddings, ids)
            return
        logger.warning("Flat indices do not support in-place updates. Consider periodic rebuilds.")

    def remove(self, ids: List[str]):
        """"in_place": tombstone the rows of the known ids (unknown ids are ignored) and return how many were removed."""
        if self.updates != "in_place":
            logger.warning("Flat indices do not support removal. Consider periodic rebuilds.")
            return
        if self.index is None:
            raise ValueError("Index not built yet")
        rows = []
        for item_id in dict.fromkeys(ids):
            row = self.reverse_id_map.pop(item_id, None)
            if row is not None:
                del self.id_map[row]
                self._set_name(row, None)
                heapq.heappush(self._free, row)
                rows.append(row)
        if rows:
            self.index.remove_rows(np.asarray(rows, dtype=np.int64))
        self.current_size = len(self.reverse_id_map)
        return len(rows)

    def _upsert(self, embeddings, ids: List[str]) -> None:
        """"in_place" add / update: known ids overwrite their rows, new ids take removed slots (lowest first), then
        append; the last occurrence of a repeated id wins."""
        embeddings = np.asarray(embeddings).astype(np.float32)
        if embeddings.ndim == 1:
            embeddings = embeddings.reshape(1, -1)
        if embeddings.ndim != 2 or embeddings.shape[1] != self.index.d or len(ids) != embeddings.shape[0]:
            raise ValueError(f"expected [len(ids) = {len(ids)}, {self.index.d}] embeddings, got {embeddings.shape}")
        last = {item_id: i for i, item_id in enumerate(ids)}
        pos = sorted(last.values())
        rows, src, tail = [], [], []
        for i in pos:
            item_id = ids[i]
            row = self.reverse_id_map.get(item_id)
            if row is None:
                if not self._free:
                    tail.append(i)
                    continue
                row = heapq.heappop(self._free)
                self.id_map[row] = item_id
                self.reverse_id_map[item_id] = row
                self._set_name(row, item_id)
            rows.append(row)
            src.append(i)
        normalize = self.metric == "cosine"
        if rows:
            self.index.update_rows(np.asarray(rows, dtype=np.int64), embeddings[src], normalize=normalize)
        if tail:
            base = self.index.ntotal
            self.index.add(embeddings[tail], normalize=normalize)
            for j, i in enumerate(tail):
                self.id_map[base + j] = ids[i]
                self.reverse_id_map[ids[i]] = base + j
            self._id_array = None
        self.current_size = len(self.reverse_id_map)
        logger.info("Upserted %d items (%d overwritten or reusing slots, %d appended). Live size: %d",
                    len(pos), len(rows), len(tail), self.current_size)

    def _drop_unmapped_rows(self) -> None:
        """"in_place" after build / load: rows no id maps to (an id given twice keeps its last row) are removed."""
        self.id_map = {row: item_id for item_id, row in sorted(self.reverse_id_map.items(), key=lambda t: t[1])}
        self._id_array = None
        dead = np.setdiff1d(np.arange(self.index.ntotal, dtype=np.int64),
                            np.fromiter(self.id_map.keys(), dtype=np.int64, count=len(self.id_map)))
        if dead.size:
            self.index.remove_rows(dead)
            self._free = dead.tolist()
            heapq.heapify(self._free)
        self.current_size = len(self.reverse_id_map)

    def compact(self) -> np.ndarray:
        """Drop removed slots on the device and renumber the id maps; returns the old -> new row map (-1 = removed)."""
        if self.index is None:
            raise ValueError("Index not built yet")
        remap = self.index.compact()
        self.id_map = {int(remap[r]): item_id for r, item_id in self.id_map.items() if remap[r] >= 0}
        self.reverse_id_map = {item_id: r for r, item_id in self.id_map.items()}
        self.current_size = len(self.reverse_id_map)
        self._free = []
        self._id_array = None
        return remap

    def save(self, path: str):
        """`<path>.faiss` = faiss' IndexFlatIP file, `<path>.pkl` = the id maps (reference retrieval.py:248-270).  Under
        "in_place" the live rows are written renumbered densely (no tombstones: a faiss reader gets a plain IndexFlatIP)
        with id maps to match."""
        if self.index is None:
            raise ValueError("No index to save")
        path = Path(path)
        path.parent.mkdir(parents=True, exist_ok=True)
        id_map, reverse_id_map, rows = self.id_map, self.reverse_id_map, self.index.reconstruct_n(0, self.index.ntotal)
        if self.updates == "in_place":
            live = np.asarray(sorted(self.id_map), dtype=np.int64)
            rows = rows[live]
            id_map = {j: self.id_map[int(r)] for j, r in enumerate(live)}
            reverse_id_map = {item_id: j for j, item_id in id_map.items()}
        write_ixfi(path.with_suffix(".faiss"), rows)
        with open(path.with_suffix(".pkl"), "wb") as f:
            pickle.dump({"id_map": id_map, "reverse_id_map": reverse_id_map,
                         "current_size": len(reverse_id_map) if self.updates == "in_place" else self.current_size,
                         "config": self.config}, f)
        logger.info("Saved index to %s", path)

    def load(self, path: str):
        """Reference retrieval.py:272-299.  Rows go back to HBM as stored (they were normalised before they were saved)."""
        path = Path(path)
        rows = read_ixfi(path.with_suffix(".faiss"))
        with open(path.with_suffix(".pkl"), "rb") as f:
            data = pickle.load(f)
        self.id_map = data["id_map"]
        self.reverse_id_map = data["reverse_id_map"]
        self._id_array = None
        self.current_size = data["current_size"]
        self.config = data["config"]
        self.dimension = rows.shape[1]
        self.index = FlatIPDeviceIndex(self.dimension, storage=self.storage)
        self.index.add(rows, normalize=False)
        self._free = []
        if self.updates == "in_place":
            self._drop_unmapped_rows()
        logger.info("Loaded index from %s with %d items", path, self.current_size)


# faiss `IxFI` file (faiss/impl/index_write.cpp, 1.7.x, what faiss.write_index emits for an IndexFlatIP,
# reference retrieval.py:261,284): fourcc "IxFI", d:int32, ntotal:int64, 2 x dummy int64 (1 << 20), is_trained:uint8,
# metric_type:int32 (0 = inner product), then the row storage as a vector<float>: count:uint64 + raw fp32 rows.
_IXFI_HEAD = "<iqqqBi"


def write_ixfi(path, rows: np.ndarray) -> None:
    rows = np.ascontiguousarray(rows, dtype=np.float32)
    if rows.ndim != 2:
        raise ValueError("write_ixfi expects a [ntotal, d] matrix")
    with open(path, "wb") as f:
        f.write(b"IxFI")
        f.write(struct.pack(_IXFI_HEAD, rows.shape[1], rows.shape[0], 1 << 20, 1 << 20, 1, 0))
        f.write(struct.pack("<Q", rows.size))
        f.write(rows.tobytes())


def read_ixfi(path) -> np.ndarray:
    with open(path, "rb") as f:
        if f.read(4) != b"IxFI":
            raise ValueError("only faiss IndexFlatIP ('IxFI') files are supported by the B200 flat index")
        d, ntotal, _, _, _, metric = struct.unpack(_IXFI_HEAD, f.read(struct.calcsize(_IXFI_HEAD)))
        if metric != 0:
            raise ValueError(f"IxFI file with metric_type {metric}: only inner product (0) is supported")
        (nfloats,) = struct.unpack("<Q", f.read(8))
        if nfloats != ntotal * d:
            raise ValueError(f"corrupt IxFI file: {nfloats} floats for {ntotal} x {d} rows")
        rows = np.frombuffer(f.read(nfloats * 4), dtype=np.float32)
        if rows.size != nfloats:
            raise ValueError("truncated IxFI file")
    return rows.reshape(ntotal, d).copy()


class RetrievalEngine:
    """The object `RecommendationService` talks to (reference retrieval.py:505-692): owns ONE index chosen by
    `config["index_type"]`, answers `retrieve(queries, k, filter_ids) -> (ids, scores, metrics)` and keeps latency
    counters.  The reference's md5 query cache is outside this hot path (SURVEY.md section 2): `use_cache` is accepted
    for signature compatibility and ignored, `cache_hit` is always False.  To keep the reference's own engine (cache
    included) and only swap the index, register `B200FlatIndex` in its `_create_index` switch — see INTEGRATION.md."""

    INDEX_TYPES = {"b200": B200FlatIndex, "faiss": B200FlatIndex}   # "faiss" configs run unchanged on the exact B200 index

    def __init__(self, config: Dict[str, Any]):
        self.config = config
        self.index_type = config.get("index_type", "b200")
        self.top_k = config.get("top_k", 100)
        self.index = self._create_index()
        self._n_calls = 0
        self._seconds = 0.0

    def _create_index(self) -> IndexBase:
        cls = self.INDEX_TYPES.get(self.index_type)
        if cls is None:
            known = self.index_type in ("annoy", "milvus")
            raise ValueError(f"index type {self.index_type!r} is not part of the B200 hot path (exact flat IP only)"
                             if known else f"Unknown index type: {self.index_type}")
        return cls({**self.config.get(self.index_type, {}), "dimension": self.config.get("embedding_dim", 128)})

    def build_index(self, embeddings: np.ndarray, ids: List[str]):
        self.index.build(embeddings, ids)

    def update_index(self, new_embeddings: np.ndarray, new_ids: List[str]):
        self.index.add(new_embeddings, new_ids)

    def account(self, seconds: float, calls: int = 1) -> None:
        """Latency bookkeeping in SECONDS (RetrievalBatcher charges one shared search to `calls` requests)."""
        self._n_calls += calls
        self._seconds += seconds

    def retrieve(self, query_embeddings, k: Optional[int] = None, filter_ids: Optional[List[str]] = None,
                 use_cache: bool = True) -> Tuple[List[List[str]], List[List[float]], Dict[str, Any]]:
        t0 = time.perf_counter()
        ids, scores = self.index.search(query_embeddings, k or self.top_k, filter_ids)
        dt = time.perf_counter() - t0
        self.account(dt)
        n = sum(map(len, ids))
        total = float(sum(sum(row) for row in scores))
        return ids, scores, {"latency_ms": dt * 1e3, "cache_hit": False, "num_results": n,
                             "avg_score": total / n if n else float("nan")}

    def get_metrics(self) -> Dict[str, Any]:
        return {"total_queries": self._n_calls, "avg_latency_ms": self._seconds / max(self._n_calls, 1) * 1e3,
                "cache_hit_rate": 0.0, "cache_size": 0, "index_size": self.index.current_size,
                "index_type": self.index_type}

    # counters under the reference's attribute names (service.py reads get_metrics(); tests may read these)
    total_queries = property(lambda self: self._n_calls)
    total_latency = property(lambda self: self._seconds)

    def save(self, path: str):
        self.index.save(path)

    def load(self, path: str):
        self.index.load(path)


def exact_topk_eval(user_emb: torch.Tensor, item_index: FlatIPDeviceIndex, train_items: Dict[int, List[int]],
                    user_rows: List[int], k: int = 100) -> np.ndarray:
    """The offline-eval twin (scripts/evaluate_model.py:217-232, src/evaluation/metrics.py:381-396): top-k item rows per
    user with that user's train items excluded, through the same fused kernel (exclusion CSR instead of a -inf mask)."""
    lists = [np.unique(np.asarray(train_items.get(u, []), dtype=np.int64)) for u in user_rows]
    indptr = np.zeros(len(lists) + 1, dtype=np.int64)
    np.cumsum([len(x) for x in lists], out=indptr[1:])
    rows = np.concatenate(lists).astype(np.int32) if indptr[-1] > 0 else np.zeros((1,), dtype=np.int32)
    dev = item_index.device
    q_op = item_index.prepare_queries(user_emb, normalize=False)
    _, ids = item_index.search_device(q_op, k, torch.from_numpy(indptr).to(dev), torch.from_numpy(rows).to(dev))
    return ids.cpu().numpy()
