"""Multi-GPU plumbing: one process per GPU, torch.distributed (NCCL over NVLink on B200; gloo in the CPU tests).

Only the two places where the hot path shards naturally use a collective (SURVEY.md section 8e):
  * retrieval: the catalogue is split row-wise, every rank scores its shard with the fused kernel (global row ids via
    row_offset), one all-gather of (score, id)[Q, k] per rank, then a k-way select on every rank;
  * data-parallel training: one all-reduce of the flat dense-gradient buffer per step.
The local search / merge callables are injectable so the world_size-2 gloo tests can exercise the partitioning and
the exchange on CPU with the oracle standing in for the CUDA kernels.
"""
from __future__ import annotations

import os

import inspect
from typing import Callable, Optional, Tuple

import numpy as np
import torch
import torch.distributed as dist


def shard_bounds(n_total: int, world: int, rank: int) -> Tuple[int, int]:
    """Contiguous row range [lo, hi) owned by `rank`: the first n_total % world ranks hold one extra row."""
    base, rem = divmod(n_total, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def shard_filter_rows(lo: int, n: int, rows=None, mask=None) -> np.ndarray:
    """Local rows (ascending, in [0, n)) of the shard that holds global rows [lo, lo + n), from a filter over GLOBAL rows:
    `rows` (int array; rows outside the shard and duplicates are dropped) or `mask` (1-D bool array over the global rows;
    a mask shorter than the catalogue leaves the missing tail not allowed, entries past the catalogue are owned by no
    shard)."""
    if (rows is None) == (mask is None):
        raise ValueError("row_filter takes exactly one of rows= or mask=")
    if mask is not None:
        m = np.asarray(mask.cpu() if torch.is_tensor(mask) else mask)
        if m.dtype != np.bool_ or m.ndim != 1:
            raise ValueError("mask must be a 1-D bool array over the global rows")
        return np.flatnonzero(m[lo: lo + n])
    r = np.asarray(rows.cpu() if torch.is_tensor(rows) else rows).reshape(-1)
    if r.size and not np.issubdtype(r.dtype, np.integer):
        raise ValueError("rows must be an integer array")
    r = r.astype(np.int64, copy=False) - lo
    return np.unique(r[(r >= 0) & (r < n)])


def shard_update_rows(lo: int, n: int, rows: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
    """(local rows, value positions) of the shard that holds global rows [lo, lo + n), from an update of GLOBAL rows
    `rows` (int64) with one value row per entry: duplicates are resolved over the whole list first (the last occurrence
    wins), then the shard keeps its own rows, ascending, and value i of its update is value positions[i] of the caller."""
    r = np.asarray(rows, dtype=np.int64).reshape(-1)
    u, first_rev = np.unique(r[::-1], return_index=True)     # ascending distinct rows, last occurrence of each
    pos = r.size - 1 - first_rev
    mine = (u >= lo) & (u < lo + n)
    return u[mine] - lo, pos[mine]


class ShardedRowFilter:
    """This rank's part of a row filter over the GLOBAL rows of a ShardedFlatIndex (`ShardedFlatIndex.row_filter`):
    `local` is the filter of the local shard (a retrieval.RowFilter over its local rows), which the shard's filtered
    sample and search steps receive.  Every rank must build it from the same global row set, as every rank passes the
    same queries; building it needs no collective."""

    def __init__(self, local):
        self.local = local


def _world() -> Tuple[int, int]:
    if dist.is_available() and dist.is_initialized():
        return dist.get_world_size(), dist.get_rank()
    return 1, 0


class _PeerExchange:
    """Symmetric (peer-mapped) gather buffers of one (batch, k) shape: every rank owns
    [thresholds: world x q x kx fp32 | scores: world x q x k fp32 | ids: world x q x k int64] and knows the address of
    its own slot inside every peer's copy, so the select kernels store their rows straight into all gather buffers over
    NVLink (b200rec_*_fanout) and the only collective left is a device-side barrier."""

    def __init__(self, group, q: int, k: int, kx: int, device):
        import torch.distributed._symmetric_memory as symm
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        pad = lambda n: (n + 255) // 256 * 256
        sec = [pad(world * q * kx * 4), pad(world * q * k * 4), pad(world * q * k * 8)]
        off = [0, sec[0], sec[0] + sec[1]]
        self.buf = symm.empty(sum(sec), dtype=torch.uint8, device=device)
        self.hdl = symm.rendezvous(self.buf, group if group is not None else dist.group.WORLD)
        base = [int(p) for p in self.hdl.buffer_ptrs]
        self.tau_dst = [base[p] + off[0] + rank * q * kx * 4 for p in range(world)]
        self.s_dst = [base[p] + off[1] + rank * q * k * 4 for p in range(world)]
        self.i_dst = [base[p] + off[2] + rank * q * k * 8 for p in range(world)]
        self.tau_all = self.buf[off[0]: off[0] + world * q * kx * 4].view(torch.float32).view(world, q, kx)
        self.s_all = self.buf[off[1]: off[1] + world * q * k * 4].view(torch.float32).view(world, q, k)
        self.i_all = self.buf[off[2]: off[2] + world * q * k * 8].view(torch.int64).view(world, q, k)

    def barrier(self, channel: int) -> None:
        self.hdl.barrier(channel=channel)


class _PeerAllReduce:
    """One-shot fp64 all-reduce of small vectors through symmetric NVLink memory (csrc/peer_reduce.cu): one 1-block
    kernel per call instead of an NCCL all-reduce (25-60 us each inside the captured training step)."""

    MAX_N = 2048

    def __init__(self, group, device):
        import ctypes
        import torch.distributed._symmetric_memory as symm
        from . import _native as N
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        if self.world > 8:
            raise RuntimeError("peer all-reduce serves one NVLink box (<= 8 ranks)")
        nbytes = int(N.lib().b200rec_peer_allreduce_bytes(self.MAX_N))
        self.buf = symm.empty((nbytes + 255) // 256 * 256, dtype=torch.uint8, device=device)
        self.buf.zero_()
        self.hdl = symm.rendezvous(self.buf, group if group is not None else dist.group.WORLD)
        self.ptrs = (ctypes.c_uint64 * self.world)(*[int(p) for p in self.hdl.buffer_ptrs])
        self.status = torch.zeros((1,), dtype=torch.int32, device=device)
        torch.cuda.synchronize(device)
        self.hdl.barrier(channel=0)          # every buffer is zeroed before anybody stores into it
        torch.cuda.synchronize(device)

    def __call__(self, t: torch.Tensor) -> None:
        from . import _native as N
        N.check(N.lib().b200rec_peer_allreduce_f64(N.ptr(t), t.numel(), self.rank, self.world, self.ptrs, self.MAX_N,
                                                   N.ptr(self.status), N.stream()), "peer_allreduce_f64")

    def check(self) -> None:
        """Raises when a call timed out waiting for a peer (synchronises: call it outside the hot step)."""
        if int(self.status.item()) != 0:
            raise RuntimeError("b200rec peer all-reduce: a replica did not answer (diverged call sequence or dead peer)")


class ShardedFlatIndex:
    """Row-sharded exact inner-product index: `search` returns the GLOBAL top-k on every rank.

    local_search(q, k, tau=None) -> (scores [Q,k] fp32, ids [Q,k] int64 with GLOBAL row ids, -1 padding)
    merge(scores [P,Q,k], ids [P,Q,k], k) -> (scores [Q,k], ids [Q,k])   order: score desc, id asc
    local_sample(q, k[, k_out, shards]) -> [Q,k_out] scores of DISTINCT local rows per query, or None (optional).  When given, shards
        all-gather these and every shard starts from the k-th best of the union: a lower bound of the GLOBAL k-th
        score, so each GPU only collects candidates that can still reach the global top-k.
    Filtered search (`search(..., sel=ShardedRowFilter)`) calls local_search(q, k, tau, out, sel=local filter) and
    local_sample(q, k, k_out, shards, sel=local filter); the filtered sampler always returns [Q,k_out] (padding rows of
    -FLT_MAX, or anything <= every real score, where it has nothing to sample).
    Live catalogue (from_device_index): `update_rows` / `remove_rows` / `compact` / `n_live` over GLOBAL rows; a shard
    with removed rows samples and searches its live rows only and, like a filtered shard, always contributes a sample.
    """

    def __init__(self, local_search: Callable, merge: Callable, group=None, local_sample: Optional[Callable] = None):
        self.local_search = local_search
        self.merge = merge
        self.group = group
        self.local_sample = local_sample
        # samplers may take (queries, k) or (queries, k, k_out, shards): the latter return k_out <= k values per query
        # from a sample thinned for `shards` pooled shards
        self._sample_takes_width = (local_sample is not None
                                    and len(inspect.signature(local_sample).parameters) >= 4)
        self.packed_exchange = False   # set by from_device_index: needs a local_search that writes into `out`
        self.peer_index = None         # set by from_device_index: the local FlatIPDeviceIndex
        self.use_peer_exchange = False # from_device_index(peer_exchange=True): fan-out stores over NVLink
        self._ids_cache = {}
        self._shard_sizes: Optional[np.ndarray] = None   # rows of every shard: gathered on the first mutation

    @classmethod
    def from_device_index(cls, index, group=None, peer_exchange: bool = True) -> "ShardedFlatIndex":
        from . import kernels as K

        def local(q_op, k, tau=None, out=None, sel=None):
            return index.search_shard(q_op, k, tau, sel=sel, out=out)

        def merge(s, i, k):
            return K.topk_merge(s, i, k)

        def sample(q_op, k, k_out=None, shards=1, sel=None):
            return index.sample_shard(q_op, k, k_out, shards, sel=sel)

        obj = cls(local, merge, group, sample)
        obj.packed_exchange = True
        obj.peer_index = index
        obj.use_peer_exchange = bool(peer_exchange)
        return obj

    def row_filter(self, rows=None, mask=None) -> ShardedRowFilter:
        """Row filter over the GLOBAL rows held now (`FlatIPDeviceIndex.row_filter` semantics: `rows` int array with
        out-of-range and duplicate rows ignored, or `mask` bool array with a missing tail not allowed; rows added later
        are not allowed).  Every rank must pass the same global set; each keeps the slice of its own shard.  Pass it as
        `sel=` to search / search_stream / search_numpy.  bf16 storage only."""
        ix = self.peer_index
        if ix is None:
            raise RuntimeError("row_filter needs a ShardedFlatIndex built by from_device_index")
        if ix.storage != "bf16":
            raise ValueError("row-sharded filtered search needs bf16 storage (the index of this shard stores fp32)")
        return ShardedRowFilter(ix.row_filter(rows=shard_filter_rows(ix.row_offset, ix.ntotal, rows, mask)))

    # ------------------------------------------------------------------ live catalogue (GLOBAL rows)
    def _local_index(self, what: str):
        if self.peer_index is None:
            raise RuntimeError(f"{what} needs a ShardedFlatIndex built by from_device_index")
        return self.peer_index

    def _all_gather(self, a: np.ndarray) -> np.ndarray:
        """Small host array of every rank -> [world, *a.shape] (one collective; outside the search path)."""
        world = dist.get_world_size(self.group)
        dev = self.peer_index.device if dist.get_backend(self.group) == "nccl" else "cpu"
        t = torch.from_numpy(np.ascontiguousarray(a).reshape(-1)).to(dev)
        out = torch.empty((world * t.numel(),), dtype=t.dtype, device=dev)
        dist.all_gather_into_tensor(out, t, group=self.group)
        return out.cpu().numpy().reshape((world,) + a.shape)

    def _global_rows(self, rows, what: str) -> np.ndarray:
        """Global rows checked against the global row count, the same on every rank (ValueError before device work)."""
        from .retrieval import check_rows
        if self._shard_sizes is None:
            self._shard_sizes = self._all_gather(np.array([self.peer_index.ntotal], np.int64))[:, 0]
        return check_rows(rows, int(self._shard_sizes.sum()), what)

    def update_rows(self, rows, x, normalize: bool = False) -> None:
        """`FlatIPDeviceIndex.update_rows` over GLOBAL rows: x[i] (host or device [n, d]) goes to global row rows[i],
        the last occurrence of a repeated row wins, a removed row is revived (how a new item takes a freed slot).  Every
        rank passes the same arguments; each copies only its shard's slice of x to its device.  No collective (except
        the one-time gather of the shard sizes); ValueError on every rank for rows outside [0, global ntotal), non-integer
        rows or a shape mismatch, before any device work."""
        ix = self._local_index("update_rows")
        if _world()[0] == 1:
            ix.update_rows(rows, x, normalize)
            return
        r = self._global_rows(rows, "update_rows")
        xt = torch.as_tensor(x)
        if xt.dim() != 2 or xt.shape[1] != ix.d or xt.shape[0] != r.size:
            raise ValueError(f"update_rows: expected [{r.size}, {ix.d}] rows, got {tuple(xt.shape)}")
        local, pos = shard_update_rows(ix.row_offset, ix.ntotal, r)
        if local.size:
            ix.update_rows(local, xt[torch.from_numpy(pos).to(xt.device)], normalize)

    def remove_rows(self, rows) -> int:
        """`FlatIPDeviceIndex.remove_rows` over GLOBAL rows; returns how many live rows were removed ON THIS SHARD.
        Every rank passes the same rows; no collective (except the one-time gather of the shard sizes)."""
        ix = self._local_index("remove_rows")
        if _world()[0] == 1:
            return ix.remove_rows(rows)
        r = self._global_rows(rows, "remove_rows")
        return ix.remove_rows(shard_filter_rows(ix.row_offset, ix.ntotal, rows=r))

    def n_live(self) -> int:
        """Live rows of the whole catalogue (one small collective: call it outside the search path)."""
        ix = self._local_index("n_live")
        if _world()[0] == 1:
            return ix.n_live
        return int(self._all_gather(np.array([ix.n_live], np.int64)).sum())

    def compact(self) -> np.ndarray:
        """Every shard drops its removed rows (rows never move between shards) and takes its new row_offset: returns the
        GLOBAL old -> new row map (int64 [old global ntotal], -1 for removed rows), the same on every rank.  Row filters
        built before are rejected afterwards; the per-shape exchange decisions are made again on the next search."""
        ix = self._local_index("compact")
        world = _world()[0]
        local = ix.compact()
        # a shard that shrank may have lost its sampling pass: the agreed ("use") and peer ("peer") choices are stale
        for key in [key for key in self._ids_cache if key[0] in ("use", "peer")]:
            del self._ids_cache[key]
        if world == 1:
            return local
        sizes = self._all_gather(np.array([local.size, ix.ntotal], np.int64))     # rows before / after, every shard
        old, new = sizes[:, 0], sizes[:, 1]
        old_off = np.concatenate([[0], np.cumsum(old)[:-1]])
        new_off = np.concatenate([[0], np.cumsum(new)[:-1]])
        ix.row_offset = int(new_off[dist.get_rank(self.group)])
        self._shard_sizes = new
        keep = np.zeros(int(old.max()), np.uint8)
        keep[: local.size] = local >= 0
        keeps = self._all_gather(keep).astype(bool)
        out = np.full(int(old.sum()), -1, np.int64)
        for p in range(world):
            kept = np.flatnonzero(keeps[p, : old[p]])
            out[old_off[p] + kept] = new_off[p] + np.arange(kept.size, dtype=np.int64)
        return out

    def _peer(self, q: int, k: int, world: int, device):
        """Peer gather buffers for this shape, or None when symmetric memory is unavailable / a shard has no sampling
        pass (then the NCCL all-gather path below runs).  Every rank takes the same branch."""
        key = ("peer", q, k)
        if key not in self._ids_cache:
            px = None
            ok = 1 if self.peer_index.has_sample_pass(q, k) else 0
            if dist.get_backend(self.group) != "nccl":
                ok = 0
            if ok:
                try:
                    px = _PeerExchange(self.group, q, k, self.exchange_width(k, world), device)
                except Exception as exc:  # noqa: BLE001 - any setup failure just selects the NCCL path
                    import logging
                    logging.getLogger("b200rec").warning("peer-memory exchange unavailable (%s): using NCCL all-gather", exc)
                    ok = 0
            flag = torch.tensor([ok], dtype=torch.int32, device=device)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.group)
            self._ids_cache[key] = px if int(flag.item()) == 1 else None
        return self._ids_cache[key]

    def _search_peer(self, px: "_PeerExchange", queries, k: int, world: int, sel=None):
        ix = self.peer_index
        # (1) sample -> every gather buffer (live and allowed rows only; padding rows where there is nothing to sample)
        ix.sample_shard(queries, k, px.tau_all.shape[2], world, sel=sel, dst=px.tau_dst)
        px.barrier(0)
        from . import kernels as K
        tau = K.topk_pooled_kth(px.tau_all, k)                                   # (2) k-th best of the pooled sample
        ix.search_shard(queries, k, tau, sel=sel, dst=(px.s_dst, px.i_dst))      # (3) local top-k -> every gather buffer
        px.barrier(1)
        return self.merge(px.s_all, px.i_all, k)                                 # (4) k-way select

    @staticmethod
    def exchange_width(k: int, world: int) -> int:
        """Sample maxima each shard contributes to the threshold exchange.  The union must hold >= k distinct rows for
        its k-th best to bound the global k-th score from below; a shard owns about k/world of the union's top k
        (binomial), so k/world + 4 sigma + 8 keeps the bound as tight as exchanging k per shard at a fraction of the
        bytes (world 8, k 100: 32 instead of 100).

        Filtered search pools the same widths, sampled over the allowed rows only, and a shard with nothing to sample
        (no allowed row, or no sampling pass for its shape) contributes padding rows of -FLT_MAX or -inf.  The bound
        still holds: if the pool holds at least k values that are scores of distinct allowed rows, its k-th best is <=
        the k-th best allowed score of the whole catalogue; if it holds fewer, its k-th best is a padding value, below
        every real score.  Padding and skew (all allowed rows on one shard, which then exchanges only k' of them) only
        loosen the bound, down to no pruning at all, so no shard has to agree with the others on whether to sample."""
        if world <= 1:
            return k
        mean = -(-k // world)
        return min(k, mean + 4 * int(mean ** 0.5) + 8)

    def _shared_thresholds(self, queries, k: int, world: int, sel=None):
        """k-th best of the union of every shard's sample: [Q] lower bounds of the global k-th score (or None).
        With a row filter `sel` (this shard's local filter): of the global k-th ALLOWED score.  Every shard then always
        contributes a [Q, k'] sample, padded where it has nothing to sample (see exchange_width), so the filtered call
        needs no agreement round."""
        kx = self.exchange_width(k, world)
        if sel is not None:
            vals = self.local_sample(queries, k, kx, world, sel=sel)
        else:
            vals = self.local_sample(queries, k, kx, world) if self._sample_takes_width else self.local_sample(queries, k)
            shape_key = ("use", int(queries.shape[0]), k)
            if shape_key not in self._ids_cache:
                # every shard must take the same branch: agree once per (batch, k) shape (one host sync, then cached)
                flag = torch.tensor([0 if vals is None else 1], dtype=torch.int32)
                if dist.get_backend(self.group) == "nccl":
                    flag = flag.cuda()
                dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.group)
                self._ids_cache[shape_key] = int(flag.item()) == 1
            if not self._ids_cache[shape_key] or vals is None:
                return None
        q, kv = vals.shape
        key = (world, q, kv, str(vals.device))
        if key not in self._ids_cache:  # any distinct ids will do: only the merged scores are used
            self._ids_cache[key] = (torch.arange(world * q * kv, dtype=torch.int64, device=vals.device).view(world, q, kv),
                                    torch.empty((world * q, kv), dtype=vals.dtype, device=vals.device))
        ids, allv = self._ids_cache[key]
        dist.all_gather_into_tensor(allv, vals.contiguous(), group=self.group)
        top, _ = self.merge(allv.view(world, q, kv), ids, k)
        return top[:, k - 1].contiguous()

    def search(self, queries, k: int, sel: Optional[ShardedRowFilter] = None):
        """Global top-k on every rank.  `sel` (from row_filter): the global exact top-k among the allowed rows, in the
        order and padding of the single-index filtered search (score desc, global row asc, -1 / -FLT_MAX past them)."""
        world, _ = _world()
        lsel = None if sel is None else sel.local
        kw = {} if sel is None else {"sel": lsel}
        if world == 1:
            if sel is None and self.peer_index is not None:   # the one-GPU search: live rows of either storage
                return self.peer_index.search_device(queries, k)
            return self.local_search(queries, k, **kw)
        if self.peer_index is not None and self.use_peer_exchange:
            px = self._peer(int(queries.shape[0]), k, world, queries.device)
            if px is not None:
                return self._search_peer(px, queries, k, world, lsel)
        tau = self._shared_thresholds(queries, k, world, lsel) if self.local_sample is not None else None
        q = int(queries.shape[0])
        if self.packed_exchange and (q * k) % 2 == 0:
            # one all-gather carries scores and ids: each rank's chunk is [q*k fp32 | q*k int64]
            dev = queries.device
            key = ("buf", q, k, str(dev))
            if key not in self._ids_cache:
                self._ids_cache[key] = (torch.empty((12 * q * k,), dtype=torch.uint8, device=dev),
                                        torch.empty((world * 12 * q * k,), dtype=torch.uint8, device=dev))
            mine, everyone = self._ids_cache[key]
            s_view = mine[: 4 * q * k].view(torch.float32).view(q, k)
            i_view = mine[4 * q * k:].view(torch.int64).view(q, k)
            self.local_search(queries, k, tau, (s_view, i_view), **kw)
            dist.all_gather_into_tensor(everyone, mine, group=self.group)
            chunks = everyone.view(world, 12 * q * k)
            gs = chunks[:, : 4 * q * k].view(torch.float32).view(world, q, k)
            gi = chunks[:, 4 * q * k:].view(torch.int64).view(world, q, k)
            return self.merge(gs, gi, k)
        if sel is not None:
            s, i = self.local_search(queries, k, tau, **kw)
        else:
            s, i = self.local_search(queries, k, tau) if tau is not None else self.local_search(queries, k)
        gs = torch.empty((world * q, s.shape[1]), dtype=s.dtype, device=s.device)
        gi = torch.empty((world * q, i.shape[1]), dtype=i.dtype, device=i.device)
        dist.all_gather_into_tensor(gs, s.contiguous(), group=self.group)
        dist.all_gather_into_tensor(gi, i.contiguous(), group=self.group)
        return self.merge(gs.view(world, q, -1), gi.view(world, q, -1), k)


    # ------------------------------------------------------------------ host-facing calls (faiss array contract)
    def _host_pipe(self, k: int, normalize: bool, share: bool, filtered: bool = False):
        from .retrieval import HostPipeline
        world, rank = _world()
        key = ("pipe", k, normalize, share, filtered)    # a filtered stream never runs the unfiltered pipe's search
        if key not in self._ids_cache:
            rows = None
            if share and world > 1:     # every replica returns the answers of ITS contiguous share of the query batch
                rows = _ShareSlice(world, rank)
            self._ids_cache[key] = HostPipeline(self.peer_index, k, normalize, lambda q_op, kk: self.search(q_op, kk), rows)
        return self._ids_cache[key]

    def search_stream(self, batches, k: int, normalize: bool = False, share_results: bool = False,
                      sel: Optional[ShardedRowFilter] = None):
        """`FlatIPDeviceIndex.search_stream` over the row-sharded catalogue: every replica passes the same HOST query
        batches (numpy) and gets faiss-shaped (D, I) numpy pairs with GLOBAL row ids.  share_results=True copies back
        only this replica's contiguous share of the queries (rows shard_bounds(nq, world, rank)), which is what a
        replicated serving tier needs; False returns the full result on every replica.  `sel` (row_filter): the exact
        top-k among the allowed rows."""
        if self.peer_index is None:
            raise RuntimeError("search_stream needs a ShardedFlatIndex built by from_device_index")
        pipe = self._host_pipe(k, normalize, share_results, sel is not None)
        if sel is not None:
            batches = self._with_filter(pipe, batches, sel)
        return self.peer_index.search_stream(batches, k, normalize, device_search=pipe)

    def _with_filter(self, pipe, batches, sel: ShardedRowFilter):
        """The batches of one filtered stream, pointing the (shared) filtered pipe's device search at `sel` right before
        each batch is submitted: every batch is searched with the filter of the stream it belongs to."""
        search = lambda q_op, kk: self.search(q_op, kk, sel=sel)   # noqa: E731
        for q in batches:
            pipe.device_search = search
            yield q

    def search_numpy(self, q, k: int, normalize: bool = False, share_results: bool = False,
                     sel: Optional[ShardedRowFilter] = None):
        """One blocking faiss-shaped call: numpy queries in, (D, I) numpy out."""
        for out in self.search_stream([q], k, normalize, share_results, sel):
            return out


class _ShareSlice:
    """slice-like: rows [lo, hi) of an nq-row batch owned by `rank` (HostPipeline calls .indices(nq))."""

    def __init__(self, world: int, rank: int):
        self.world, self.rank = world, rank

    def indices(self, nq: int):
        lo, hi = shard_bounds(nq, self.world, self.rank)
        return lo, hi, 1


class _AllGatherRows(torch.autograd.Function):
    """x [B,E] on every replica -> [world*B, E] (rank-major); backward = reduce-scatter (sum) of the gathered gradient."""

    @staticmethod
    def forward(ctx, x, group):
        ctx.group = group
        x = x.contiguous()
        out = torch.empty((dist.get_world_size(group) * x.shape[0], x.shape[1]), dtype=x.dtype, device=x.device)
        dist.all_gather_into_tensor(out, x, group=group)
        return out

    @staticmethod
    def backward(ctx, g):
        world = dist.get_world_size(ctx.group)
        rows = g.shape[0] // world
        if dist.get_backend(ctx.group) == "gloo":   # CPU tests: gloo has no reduce-scatter
            total = g.contiguous().clone()
            dist.all_reduce(total, op=dist.ReduceOp.SUM, group=ctx.group)
            r = dist.get_rank(ctx.group)
            return total[r * rows:(r + 1) * rows].clone(), None
        gx = torch.empty((rows, g.shape[1]), dtype=g.dtype, device=g.device)
        dist.reduce_scatter_tensor(gx, g.contiguous(), op=dist.ReduceOp.SUM, group=ctx.group)
        return gx, None


class _TowerDP:
    """The data-parallel context one tower sees: everything of the parent DataParallel, but its own peer all-reduce
    buffers.  The call sequence of a peer all-reduce context must be identical on every replica; with one context per
    tower the two towers can run on different streams (their kernels interleave differently on every GPU)."""

    def __init__(self, parent: "DataParallel", peer_ar):
        self._parent, self._peer_ar = parent, peer_ar

    def __getattr__(self, name):
        if name.startswith("_"):   # copy / pickle probe dunder and private names before __init__ has run
            raise AttributeError(name)
        return getattr(self._parent, name)

    def reduce_sums(self, t: torch.Tensor) -> None:
        DataParallel._reduce_small(self._peer_ar, self._parent.group, t)


class DataParallel:
    """Exact data-parallel training of the two-tower model (one process per GPU, equal local batches): the result is
    what ONE process computes on the concatenated global batch (reference trainers/two_tower.py:98-151):
      * BatchNorm batch statistics over all replicas (fp64 partial sums all-reduced inside b200rec_bn_*_dp);
      * in-batch negatives = the all-gathered item embeddings of the global batch, gradients reduce-scattered back;
      * losses normalised by the GLOBAL batch, so gradients are SUMMED: one all-reduce of the flat dense gradient buffer
        and an all-gather + re-coalesce of the touched rows of row-sparse embedding tables."""

    def __init__(self, model, group=None):
        if not (dist.is_available() and dist.is_initialized()):
            raise RuntimeError("DataParallel needs an initialised torch.distributed process group")
        self.group = group
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        model.dp = self
        model.user_tower.dp = self
        model.item_tower.dp = self
        # Dense id-embedding tables: a step's gradient is non-zero on the rows the GLOBAL batch touched only, so the
        # replicas exchange (ids, gradient rows) of their samples (world x B x (8 + 4e) bytes) and every replica adds all
        # of them into its own dense gradient — the same sum an all-reduce of the whole [rows, e] buffer would produce
        # (282 MB per step for config 2), see ops.GatherConcatFn.backward and FlatAdam.step.
        for tower in (model.user_tower, model.item_tower):
            for emb in getattr(tower, "embeddings", {}).values():
                if not getattr(emb.weight, "_b200_sparse", False):
                    emb.weight._b200_row_exchange = self
        self._setup_peer_allreduce(model)

    def _setup_peer_allreduce(self, model) -> None:
        """NVLink peer-memory all-reduce for the small fp64 exchanges (BatchNorm sums, loss): every rank takes the same
        branch (agreed with one MIN all-reduce); anything that fails selects the NCCL path."""
        self._peer_ar = None
        self.streams_safe = False
        if os.environ.get("B200REC_PEER_ALLREDUCE", "1") == "0" or dist.get_backend(self.group) != "nccl":
            return
        dev = next(model.parameters()).device
        ctx, ok = [], 1
        try:
            ctx = [_PeerAllReduce(self.group, dev) for _ in range(3)]   # loss / user tower / item tower
        except Exception as exc:  # noqa: BLE001
            import logging
            logging.getLogger("b200rec").warning("peer-memory all-reduce unavailable (%s): using NCCL", exc)
            ok = 0
        flag = torch.tensor([ok], dtype=torch.int32, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.group)
        if int(flag.item()) != 1:
            return
        self._peer_ar = ctx[0]
        model.user_tower.dp = _TowerDP(self, ctx[1])
        model.item_tower.dp = _TowerDP(self, ctx[2])
        # no collective of a tower goes through the (single, ordered) NCCL communicator any more except the touched-row
        # exchange, which torch orders by host call: the towers may run on two streams as they do on one GPU
        self.streams_safe = os.environ.get("B200REC_DP_OVERLAP", "1") != "0"

    @staticmethod
    def _reduce_small(pr, group, t: torch.Tensor) -> None:
        if (pr is not None and t.dtype == torch.float64 and t.is_cuda and t.is_contiguous()
                and 0 < t.numel() <= pr.MAX_N):
            pr(t)
            return
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)

    def reduce_sums(self, t: torch.Tensor) -> None:
        """In-place sum over the replicas of a small statistics vector (fp64 BatchNorm sums): bit-identical everywhere."""
        self._reduce_small(getattr(self, "_peer_ar", None), self.group, t)

    def all_gather_rows(self, x: torch.Tensor) -> torch.Tensor:
        return _AllGatherRows.apply(x, self.group)

    def reduce_dense_grad_(self, flat: torch.Tensor, runs=None) -> None:
        """Sum the flat gradient buffer over the replicas; `runs` = [lo, hi) element ranges to reduce (default: all)."""
        if runs is None:
            dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=self.group)
            return
        for lo, hi in runs:
            dist.all_reduce(flat[lo:hi], op=dist.ReduceOp.SUM, group=self.group)

    def gather_sparse(self, rows: torch.Tensor, vals: torch.Tensor):
        """(rows [n] int64, vals [n,e] fp32) of this replica -> concatenation over replicas (padding rows stay 0).
        ONE collective: the ids travel as two extra fp32 columns (bit pattern) of the value rows."""
        n, e = vals.shape
        packed = torch.empty((n, e + 2), dtype=torch.float32, device=vals.device)
        packed[:, :e] = vals
        packed[:, e:] = rows.contiguous().view(torch.float32).view(n, 2)
        everyone = torch.empty((self.world * n, e + 2), dtype=torch.float32, device=vals.device)
        dist.all_gather_into_tensor(everyone, packed, group=self.group)
        ar = everyone[:, e:].contiguous().view(torch.int64).view(-1)
        av = everyone[:, :e].contiguous()
        return ar, av

    def gather_counts(self, n: int):
        """[n of every replica] (host ints; one small collective, used outside the hot step)."""
        dev = "cuda" if dist.get_backend(self.group) == "nccl" else "cpu"
        t = torch.zeros((self.world,), dtype=torch.int64, device=dev)
        t[self.rank] = int(n)
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)
        return [int(x) for x in t.tolist()]

    def global_loss(self, local_share: torch.Tensor) -> torch.Tensor:
        if getattr(self, "_peer_ar", None) is not None and local_share.is_cuda:
            out = local_share.detach().to(torch.float64).reshape(1)
            self.reduce_sums(out)
            return out.to(local_share.dtype).reshape(local_share.shape)
        out = local_share.detach().clone()
        dist.all_reduce(out, op=dist.ReduceOp.SUM, group=self.group)
        return out
