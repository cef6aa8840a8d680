"""CPU checks of row-sharded filtered search (ShardedFlatIndex.row_filter / search(sel=)): slicing a filter over GLOBAL
rows into each shard's local rows, and a world_size-2 gloo run of the filtered exchange with the oracle standing in for
the CUDA sample / search steps, against the oracle over the allowed rows alone."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def oracle_allowed(xb, q, k, mask):
    """Exact top-k over the rows where `mask` is True (the oracle over those rows alone, ids mapped back through the
    ascending row list, so the (score desc, row asc) order is kept); -1 / -FLT_MAX padding."""
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


def test_global_rows_are_sliced_into_shard_local_rows():
    from b200rec.dist import shard_bounds, shard_filter_rows
    N, world = 1003, 3                                           # uneven shards: 335, 334, 334 rows
    spans = [shard_bounds(N, world, r) for r in range(world)]
    assert [h - l for l, h in spans] == [335, 334, 334]
    rows = np.array([-5, 0, 334, 335, 335, 668, 669, 1002, 1003, 5000, 700, 700, 336])
    want = {0: [0, 334], 1: [0, 1, 333], 2: [0, 31, 333]}
    for r, (lo, hi) in enumerate(spans):
        got = shard_filter_rows(lo, hi - lo, rows=rows)
        assert got.dtype == np.int64 and got.tolist() == want[r]                 # ascending, deduplicated, in range
        assert shard_filter_rows(lo, hi - lo, rows=rows.astype(np.int32)).tolist() == want[r]
    mask = np.zeros(N, bool)
    mask[rows[(rows >= 0) & (rows < N)]] = True
    for r, (lo, hi) in enumerate(spans):
        assert shard_filter_rows(lo, hi - lo, mask=mask).tolist() == want[r]
    short = mask[:400]                                          # the missing tail is not allowed
    assert shard_filter_rows(0, 335, mask=short).tolist() == [0, 334]
    assert shard_filter_rows(spans[1][0], 334, mask=short).tolist() == [0, 1]
    assert shard_filter_rows(spans[2][0], 334, mask=short).tolist() == []
    assert shard_filter_rows(0, 10, rows=np.array([], np.int64)).tolist() == []
    with pytest.raises(ValueError, match="exactly one"):
        shard_filter_rows(0, 10)
    with pytest.raises(ValueError, match="exactly one"):
        shard_filter_rows(0, 10, rows=[1], mask=np.ones(10, bool))
    with pytest.raises(ValueError, match="integer"):
        shard_filter_rows(0, 10, rows=np.array([1.5]))
    with pytest.raises(ValueError, match="bool"):
        shard_filter_rows(0, 10, mask=np.ones(10, np.int8))


def _cases(N, spans, k, rng):
    """name -> (global mask, rank whose sample is padding only or None, pass as rows= instead of mask=)."""
    (lo0, hi0), (lo1, hi1) = spans
    one = np.zeros(N, bool)
    one[lo1 + rng.permutation(hi1 - lo1)[:300]] = True                         # every allowed row on shard 1
    few = np.zeros(N, bool)
    few[rng.permutation(N)[: k - 7]] = True                                      # fewer than k allowed rows in all
    uni = rng.random(N) < 0.2
    return {"all on one shard (shard 0 empty)": (one, None, True),
            "fewer than k allowed": (few, None, False),
            "shard 0 samples padding only": (uni, 0, True),
            "both shards sample padding only": (uni, -1, False),
            "empty filter": (np.zeros(N, bool), None, False),
            "every row": (np.ones(N, bool), None, True)}


def _gloo_worker(rank, world, port, tmp):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    from b200rec.dist import ShardedFlatIndex, ShardedRowFilter, shard_bounds, shard_filter_rows
    from oracle.flat_ip import FLT_MAX, IndexFlatIP, merge_topk
    dist.init_process_group("gloo", rank=rank, world_size=world)
    rng = np.random.default_rng(8)
    N, Q, D, k = 4001, 29, 12, 40
    cat = rng.integers(-2, 3, size=(N, D)).astype(np.float32)     # integer data: exact sums, massive ties
    qry = rng.integers(-2, 3, size=(Q, D)).astype(np.float32)
    spans = [shard_bounds(N, world, r) for r in range(world)]
    lo, hi = spans[rank]
    pad_rank = {"rank": None}

    def local_rows_search(rows, q, kk):
        s = np.full((len(q), kk), -FLT_MAX, np.float32)
        i = np.full((len(q), kk), -1, np.int64)
        if rows.size:
            ix = IndexFlatIP(D)
            ix.add(cat[lo + rows])
            s, j = ix.search(q, kk)
            i = np.where(j >= 0, lo + rows[np.maximum(j, 0)], -1)
        return s, i

    def local(q, kk, tau=None, out=None, sel=None):            # the oracle stands in for the filtered shard search
        s, i = local_rows_search(sel, q, kk)
        if tau is not None:                                     # the pooled threshold drops what cannot reach the top-k
            drop = s < tau.numpy()[:, None]
            s, i = np.where(drop, -FLT_MAX, s), np.where(drop, -1, i)
        return torch.from_numpy(s.astype(np.float32)), torch.from_numpy(i)

    def sample(q, kk, k_out=None, shards=1, sel=None):          # any distinct allowed rows: the first 150 of the shard
        if pad_rank["rank"] in (rank, -1):
            return torch.full((len(q), k_out), -FLT_MAX, dtype=torch.float32)
        s, _ = local_rows_search(sel[:150], q, k_out)
        return torch.from_numpy(s)

    def merge(s, i, kk):
        ms, mi = merge_topk([s[p].numpy() for p in range(s.shape[0])], [i[p].numpy() for p in range(i.shape[0])], kk)
        return torch.from_numpy(ms), torch.from_numpy(mi)

    sh = ShardedFlatIndex(local, merge, local_sample=sample)
    thresholds = {}
    orig = sh._shared_thresholds

    def spy(queries, kk, w, sel=None):
        tau = orig(queries, kk, w, sel)
        thresholds["tau"] = tau
        return tau
    sh._shared_thresholds = spy
    lines = []
    for name, (mask, pad, as_rows) in _cases(N, spans, k, rng).items():
        pad_rank["rank"] = pad
        if as_rows:   # global rows with duplicates and out-of-range rows, which the filter ignores
            g = np.flatnonzero(mask)
            loc = shard_filter_rows(lo, hi - lo, rows=np.concatenate([g, g[:9], [-1, N, N + 50]]))
        else:
            loc = shard_filter_rows(lo, hi - lo, mask=mask)
        s, i = sh.search(qry, k, sel=ShardedRowFilter(loc))
        rD, rI = oracle_allowed(cat, qry, k, mask)
        tau = thresholds["tau"].numpy()
        ok = (np.array_equal(i.numpy(), rI) and np.array_equal(s.numpy(), rD) and (tau <= rD[:, k - 1]).all()
              and (pad != -1 or (tau == -FLT_MAX).all()))
        lines.append(f"{name}: {int(ok)}")
    with open(os.path.join(tmp, f"ok{rank}"), "w") as fh:
        fh.write("\n".join(lines))
    dist.destroy_process_group()


def test_sharded_filtered_search_world_size_2_gloo(tmp_path):
    """Both shards pass the same global filter; each keeps its slice.  Every case must equal the oracle over the allowed
    rows alone, bit for bit, with a pooled threshold <= the k-th allowed score: all allowed rows on one shard (the other
    has none), fewer than k allowed rows in all, a shard (or both) contributing a sample of padding only, an empty filter
    and an all-allowed one."""
    import torch.multiprocessing as mp
    port = 31500 + (os.getpid() % 2000)
    mp.spawn(_gloo_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    for r in range(2):
        lines = open(tmp_path / f"ok{r}").read().splitlines()
        assert len(lines) == 6 and all(l.endswith(": 1") for l in lines), (r, lines)
