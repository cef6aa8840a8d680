"""CPU checks of the live catalogue on the row-sharded index (ShardedFlatIndex.update_rows / remove_rows / compact /
n_live over GLOBAL rows): slicing updates and removals into each shard's local rows, and a world_size-2 gloo run with an
oracle-backed stand-in for each rank's FlatIPDeviceIndex, so the partitioning, the validation, the exchange (through the
closures of from_device_index) and compact()'s global row map are exercised against the oracle over the live rows."""
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_global_updates_and_removals_are_sliced_into_shard_local_rows():
    from b200rec.dist import shard_bounds, shard_filter_rows, shard_update_rows
    N, world = 1003, 3                                           # uneven shards: 335, 334, 334 rows
    spans = [shard_bounds(N, world, r) for r in range(world)]
    rows = np.array([334, 335, 334, 668, 669, 0, 335, 1002, 668, 700])
    # last occurrence per row: 334 -> 2, 335 -> 6, 668 -> 8, 669 -> 4, 0 -> 5, 1002 -> 7, 700 -> 9
    want = {0: ([0, 334], [5, 2]), 1: ([0, 333], [6, 8]), 2: ([0, 31, 333], [4, 9, 7])}
    for r, (lo, hi) in enumerate(spans):
        local, pos = shard_update_rows(lo, hi - lo, rows)
        assert local.dtype == np.int64 and pos.dtype == np.int64
        assert (local.tolist(), pos.tolist()) == want[r], r
        assert shard_filter_rows(lo, hi - lo, rows=rows).tolist() == want[r][0]   # removals: the same rows, no values
    for r, (lo, hi) in enumerate(spans):
        local, pos = shard_update_rows(lo, hi - lo, np.zeros(0, np.int64))
        assert local.size == 0 and pos.size == 0


def oracle_live(xb, q, k, mask):
    """Exact top-k over the rows where `mask` is True, ids mapped back through the ascending row list; padding."""
    from oracle.flat_ip import FLT_MAX, IndexFlatIP
    rows = np.flatnonzero(mask)
    D = np.full((len(q), k), -FLT_MAX, np.float32)
    I = np.full((len(q), k), -1, np.int64)
    if rows.size:
        ix = IndexFlatIP(xb.shape[1])
        ix.add(xb[rows])
        D, i = ix.search(q, k)
        I = np.where(i >= 0, rows[np.maximum(i, 0)], -1)
    return D, I


class _Filter:
    def __init__(self, rows, generation):
        self.rows, self.generation = rows, generation


class _OracleShard:
    """CPU stand-in for one rank's FlatIPDeviceIndex in HOST-LOGIC tests only: local row slots + live mask, with the
    sample_shard / search_shard steps answered by the oracle over the live (and allowed) rows, global ids."""

    storage = "bf16"

    def __init__(self, xb, row_offset):
        import torch
        self.d = xb.shape[1]
        self.device = torch.device("cpu")
        self.xb = xb.copy()
        self.live = np.ones(len(xb), bool)
        self.row_offset = row_offset
        self.generation = 0
        self.calls = []

    ntotal = property(lambda self: len(self.xb))
    n_live = property(lambda self: int(self.live.sum()))

    def update_rows(self, rows, x, normalize=False):
        rows = np.asarray(rows)
        assert rows.dtype == np.int64 and len(set(rows.tolist())) == len(rows) and ((rows >= 0) & (rows < self.ntotal)).all()
        self.calls.append(("update_rows", len(rows)))
        self.xb[rows] = np.asarray(x, np.float32)
        self.live[rows] = True

    def remove_rows(self, rows):
        rows = np.unique(np.asarray(rows, np.int64))
        assert ((rows >= 0) & (rows < self.ntotal)).all()
        if rows.size == 0:
            return 0
        self.calls.append(("remove_rows", len(rows)))
        n = int(self.live[rows].sum())
        self.live[rows] = False
        return n

    def compact(self):
        keep = np.flatnonzero(self.live)
        remap = np.full(self.ntotal, -1, np.int64)
        remap[keep] = np.arange(keep.size)
        self.xb, self.live = self.xb[keep], np.ones(keep.size, bool)
        self.generation += 1
        return remap

    def row_filter(self, rows=None, mask=None):
        return _Filter(np.asarray(rows, np.int64), self.generation)

    def has_sample_pass(self, nq, k):
        return True

    def _mask(self, sel):
        m = self.live.copy()
        if sel is not None:
            if sel.generation != self.generation:
                raise ValueError("the row filter was built before compact() renumbered the rows; build it again")
            allowed = np.zeros(self.ntotal, bool)
            allowed[sel.rows] = True
            m &= allowed
        return m

    def sample_shard(self, q, k, k_out=None, shards=1, sel=None, dst=None):
        import torch
        m = self._mask(sel)
        m[np.flatnonzero(m)[150:]] = False                      # any distinct live allowed rows: the first 150
        s, _ = oracle_live(self.xb, q.numpy(), k if k_out is None else k_out, m)
        return torch.from_numpy(s)

    def search_shard(self, q, k, tau, sel=None, out=None, dst=None):
        import torch
        from oracle.flat_ip import FLT_MAX
        s, i = oracle_live(self.xb, q.numpy(), k, self._mask(sel))
        i = np.where(i >= 0, i + self.row_offset, -1)
        if tau is not None:                                      # the pooled threshold drops what cannot reach the top-k
            drop = s < tau.numpy()[:, None]
            s, i = np.where(drop, -FLT_MAX, s).astype(np.float32), np.where(drop, -1, i)
        s, i = torch.from_numpy(s), torch.from_numpy(i)
        if out is not None:
            out[0].copy_(s)
            out[1].copy_(i)
            return out
        return s, i


def _gloo_worker(rank, world, port, tmp):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    from b200rec.dist import ShardedFlatIndex, shard_bounds
    from oracle.flat_ip import merge_topk
    dist.init_process_group("gloo", rank=rank, world_size=world)
    rng = np.random.default_rng(9)                              # same seed on every rank: same global calls
    N, Q, D = 4001, 29, 12
    cat = rng.integers(-2, 3, size=(N, D)).astype(np.float32)   # integer data: exact sums, massive ties
    qry = rng.integers(-2, 3, size=(Q, D)).astype(np.float32)
    qt = torch.from_numpy(qry)
    live = np.ones(N, bool)
    lo, hi = shard_bounds(N, world, rank)
    shard = _OracleShard(cat[lo:hi], lo)
    sh = ShardedFlatIndex.from_device_index(shard, peer_exchange=False)

    def merge(s, i, kk):
        ms, mi = merge_topk([s[p].numpy() for p in range(s.shape[0])], [i[p].numpy() for p in range(i.shape[0])], kk)
        return torch.from_numpy(ms), torch.from_numpy(mi)
    sh.merge = merge
    out = {"errors": [], "checks": []}

    def check(name, mask, sel=None):
        for k in (40, 41):                                      # Q * k even: packed all-gather; odd: two all-gathers
            s, i = sh.search(qt, k, sel=sel)
            rD, rI = oracle_live(cat, qry, k, mask)
            out["checks"].append([f"{name} k={k}", bool(np.array_equal(i.numpy(), rI) and np.array_equal(s.numpy(), rD))])

    # validation: the same ValueError on every rank, before any device work
    x2 = np.zeros((2, D), np.float32)
    for bad in ([3, N], [-1, 2], np.array([1.0, 2.0]), np.array([[1, 2]])):
        for call in (lambda: sh.update_rows(bad, x2), lambda: sh.remove_rows(bad)):
            with pytest.raises(ValueError) as e:
                call()
            out["errors"].append(str(e.value))
    for shape in ((3, D), (2, D + 1), (2,)):
        with pytest.raises(ValueError) as e:
            sh.update_rows([1, 2], np.zeros(shape, np.float32))
        out["errors"].append(str(e.value))
    out["no_device_call"] = shard.calls == []
    out["sizes"] = sh._shard_sizes.tolist()

    sel_mask = rng.random(N) < 0.4
    sel = sh.row_filter(mask=sel_mask)                          # built before the mutations
    check("unmutated", live)
    removed_here = []
    for rnd in range(5):                                        # update (duplicates across the boundary) / remove / revive
        rows = rng.integers(0, N, size=300)
        rows[:20] = shard_bounds(N, world, 0)[1] - 10 + np.arange(20)          # straddle the shard boundary
        rows[20:40] = rows[:20][::-1]                                          # duplicates: the later value wins
        dead = np.flatnonzero(~live)[:30]
        rows[rows.size - dead.size:] = dead                                    # revive removed rows
        x = rng.integers(-2, 3, size=(rows.size, D)).astype(np.float32)
        sh.update_rows(rows, x)
        for r, v in zip(rows, x):
            cat[r] = v
        live[rows] = True
        rm = rng.integers(0, N, size=(5, 400, 1500, 40, 10)[rnd])
        rm = np.concatenate([rm, rm[:3], np.flatnonzero(~live)[:3]])
        u = np.unique(rm)
        mine = u[(u >= lo) & (u < hi)]
        removed_here.append(sh.remove_rows(rm) == int(live[mine].sum()))
        live[rm] = False
        out["checks"].append([f"n_live round {rnd}", sh.n_live() == int(live.sum())])
        check(f"round {rnd}", live)
        check(f"filter round {rnd}", live & sel_mask, sel)
    out["checks"].append(["remove_rows counts this shard", all(removed_here)])
    # a shard with every row removed pads; then fewer than k live rows in all
    lo0, hi0 = shard_bounds(N, world, 0)
    sh.remove_rows(np.arange(lo0, hi0))
    live[lo0:hi0] = False
    check("shard 0 empty", live)
    keep = np.flatnonzero(live)[:25]
    sh.remove_rows(np.setdiff1d(np.flatnonzero(live), keep))
    live[:] = False
    live[keep] = True
    check("fewer than k live", live)
    revive = np.array([lo0 + 3, lo0 + 5, hi0 - 1, hi0])          # freed slots take new items, on both shards
    xr = rng.integers(-2, 3, size=(revive.size, D)).astype(np.float32)
    sh.update_rows(revive, xr)
    cat[revive] = xr
    live[revive] = True
    check("revived", live)
    out["cached_use_before"] = any(key[0] == "use" for key in sh._ids_cache)
    bD, bI = sh.search(qt, 40)
    remap = sh.compact()
    out["remap"] = remap.tolist()
    out["row_offset"] = shard.row_offset
    out["cached_use_after"] = any(key[0] in ("use", "peer") for key in sh._ids_cache)
    aD, aI = sh.search(qt, 40)
    out["checks"].append(["compact keeps results", bool(np.array_equal(aD.numpy(), bD.numpy()) and np.array_equal(
        aI.numpy(), np.where(bI.numpy() >= 0, remap[np.maximum(bI.numpy(), 0)], -1)))])
    cat, live = cat[live], np.ones(int(live.sum()), bool)
    check("after compact", live)
    out["checks"].append(["n_live after compact", sh.n_live() == live.size])
    with pytest.raises(ValueError, match="compact"):
        sh.search(qt, 40, sel=sel)
    out["stale_filter_rejected"] = True
    with pytest.raises(ValueError):                              # the global row count was refreshed
        sh.remove_rows([live.size])
    sh.remove_rows([live.size - 1])
    live[-1] = False
    check("after compact, mutated again", live)
    with open(os.path.join(tmp, f"out{rank}.json"), "w") as fh:
        json.dump(out, fh)
    dist.destroy_process_group()


def test_sharded_live_catalogue_world_size_2_gloo(tmp_path):
    """Both ranks pass the same global calls.  Bad arguments raise the same ValueError on both ranks with no device call;
    random update / remove / revive rounds (updates straddling the shard boundary, duplicates, revived slots) and a
    filter built before them equal the oracle over the live rows bit for bit on both exchange forms; a shard with every
    row removed pads; compact() returns the same global map on both ranks, moves rank 1's offset, drops the cached
    exchange decisions and rejects the old filter."""
    import torch.multiprocessing as mp
    port = 33500 + (os.getpid() % 2000)
    mp.spawn(_gloo_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    outs = [json.load(open(tmp_path / f"out{r}.json")) for r in range(2)]
    for r, o in enumerate(outs):
        bad = [name for name, ok in o["checks"] if not ok]
        assert not bad and len(o["checks"]) >= 30, (r, bad)
        assert o["no_device_call"] and o["stale_filter_rejected"], r
        assert o["sizes"] == [2001, 2000]
        assert o["cached_use_before"] and not o["cached_use_after"], r
    assert outs[0]["errors"] == outs[1]["errors"] and len(outs[0]["errors"]) == 11
    assert outs[0]["remap"] == outs[1]["remap"] and len(outs[0]["remap"]) == 4001
    remap = np.asarray(outs[0]["remap"])
    kept = np.flatnonzero(remap >= 0)
    assert np.array_equal(remap[kept], np.arange(kept.size))     # live rows keep their order, densely renumbered
    assert outs[0]["row_offset"] == 0 and outs[1]["row_offset"] == int((remap[:2001] >= 0).sum())
