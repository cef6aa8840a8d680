"""GPU parity of row-sharded filtered search: unequal row shards emulated on one GPU run the steps every rank runs —
filtered sample (allowed rows only, padding where a shard has nothing to sample), pooled k-th, filtered search from that
threshold, k-way merge — with each shard forced onto the bitmap or the compacted path, against the CPU oracle over the
allowed rows alone, bit for bit on integer data with massive ties; the fan-out entry points against the plain calls; the
host-facing calls of ShardedFlatIndex on one GPU; and, on two GPUs, tools/check_sharded_filtered.py over both
exchange paths."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

SPANS = ((0, 40_000), (40_000, 110_000), (110_000, 200_000))   # unequal shards of a 200 K-row catalogue
PATHS = ((False, False, False), (True, True, True), (False, True, False), (True, False, True))   # compact per shard


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


def _int_shards(cat, spans=SPANS):
    from b200rec.retrieval import FlatIPDeviceIndex
    shards = []
    for lo, hi in spans:
        ix = FlatIPDeviceIndex(cat.shape[1], storage="bf16", row_offset=lo)
        ix.add(cat[lo:hi])
        shards.append(ix)
    return shards


def _int_data(N, D, Q, seed, lo=-2, hi=3):
    rng = np.random.default_rng(seed)
    cat = rng.integers(lo, hi, size=(N, D)).astype(np.float32)        # bf16-exact values, exact fp32 sums: massive ties
    qry = rng.integers(lo, hi, size=(Q, D)).astype(np.float32)
    return cat, qry, rng


def _local_filters(shards, mask):
    from b200rec.dist import shard_filter_rows
    return [ix.row_filter(rows=shard_filter_rows(ix.row_offset, ix.ntotal, mask=mask)) for ix in shards]


def _sharded(shards, q_op, k, sels, paths):
    """What every rank runs, with the exchange done on one device: (tau [Q], D [Q,k], I [Q,k])."""
    from b200rec import kernels as KR
    from b200rec.dist import ShardedFlatIndex
    world = len(shards)
    kx = ShardedFlatIndex.exchange_width(k, world)
    vals = torch.stack([ix.sample_filtered(q_op, k, kx, world, sel, compact=c)
                        for ix, sel, c in zip(shards, sels, paths)]).contiguous()
    tau = KR.topk_pooled_kth(vals, k)
    parts = [ix.search_filtered_shard(q_op, k, sel, tau, compact=c) for ix, sel, c in zip(shards, sels, paths)]
    D, I = KR.topk_merge(torch.stack([p[0] for p in parts]).contiguous(), torch.stack([p[1] for p in parts]).contiguous(), k)
    return tau.cpu().numpy(), D.cpu().numpy(), I.cpu().numpy()


def _filters(N, rng):
    lo1, hi1 = SPANS[1]
    out = {"empty": np.zeros(N, bool)}
    one = np.zeros(N, bool)
    one[lo1 + rng.permutation(hi1 - lo1)[: (hi1 - lo1) // 20]] = True
    out["all on shard 1"] = one
    skip0 = rng.random(N) < 0.1
    skip0[: SPANS[0][1]] = False
    out["shard 0 empty"] = skip0
    for f in (0.001, 0.1, 0.5, 1.0):
        m = np.zeros(N, bool)
        m[rng.permutation(N)[: int(round(f * N))]] = True
        out[f"random {f:g}"] = m
    return out


@pytest.mark.parametrize("Q,k", [(300, 10), (300, 100), (300, 1000), (40, 10), (40, 100), (40, 1000)])
def test_emulated_shards_equal_the_oracle_bit_for_bit(Q, k):
    """Q >= 256 runs the CTA-pair kernel, Q < 256 the single-CTA one.  k = 1000 has no sampling pass (every shard pools
    padding: no pruning); at k = 10 / 100 the 40 K-row shard and small compacted operands have none either."""
    cat, qry, rng = _int_data(SPANS[-1][1], 64, Q, seed=Q + k)
    shards = _int_shards(cat)
    q_op = shards[0].prepare_queries(qry)
    for name, mask in _filters(cat.shape[0], rng).items():
        sels = _local_filters(shards, mask)
        rD, rI = oracle_allowed(cat, qry, k, mask)
        for paths in PATHS:
            tau, D, I = _sharded(shards, q_op, k, sels, paths)
            assert np.array_equal(I, rI), (name, paths)
            assert np.array_equal(D, rD), (name, paths)
            assert (tau <= rD[:, k - 1]).all(), (name, paths)


@pytest.mark.parametrize("Q", [300, 40])
def test_pooled_threshold_respects_the_filter_on_every_shard(Q):
    """Every disallowed row outscores every allowed row, on every shard: a shard whose sample ignored the filter would
    pool a threshold above every allowed score and the search would return nothing."""
    N, D, k = SPANS[-1][1], 64, 100
    rng = np.random.default_rng(Q)
    mask = rng.random(N) < 0.3
    cat = rng.integers(1, 3, size=(N, D)).astype(np.float32)
    cat[mask] = -rng.integers(1, 3, size=(int(mask.sum()), D)).astype(np.float32)
    qry = rng.integers(1, 3, size=(Q, D)).astype(np.float32)
    shards = _int_shards(cat)
    assert all(ix.has_sample_pass(Q, k) for ix in shards[1:])
    q_op = shards[0].prepare_queries(qry)
    sels = _local_filters(shards, mask)
    rD, rI = oracle_allowed(cat, qry, k, mask)
    assert (rD < 0).all() and (rI >= 0).all()
    for paths in PATHS:
        tau, D_, I_ = _sharded(shards, q_op, k, sels, paths)
        assert (tau <= rD[:, k - 1]).all(), paths
        if not any(paths[1:]):      # two bitmap shards pool 2 x 62 >= k real values (one alone pools padding)
            assert (tau > -3.0e38).any(), paths
        assert np.array_equal(I_, rI) and np.array_equal(D_, rD), paths


def test_fanout_entry_points_equal_the_plain_calls():
    """Two local destinations stand in for two peers' gather buffers: both receive exactly what the plain call returns,
    for the masked sample, the bitmap search, the compact search (ids mapped inside the select kernel) and a shard with
    no allowed row (padding stored to every destination)."""
    from b200rec.dist import ShardedFlatIndex
    Q, k = 300, 100
    cat, qry, rng = _int_data(SPANS[-1][1], 64, Q, seed=5)
    shards = _int_shards(cat)
    q_op = shards[0].prepare_queries(qry)
    mask = rng.random(cat.shape[0]) < 0.2
    mask[: SPANS[0][1]] = False                                           # shard 0 has no allowed row
    sels = _local_filters(shards, mask)
    kx = ShardedFlatIndex.exchange_width(k, 3)
    tau = torch.full((Q,), 4.0, device="cuda")
    for ix, sel in zip(shards, sels):
        for compact in (False, True):
            plain = ix.sample_filtered(q_op, k, kx, 3, sel, compact=compact)
            dst = [torch.full((Q, kx), float("nan"), device="cuda") for _ in range(2)]
            assert ix.sample_filtered(q_op, k, kx, 3, sel, dst=[t.data_ptr() for t in dst], compact=compact) is None
            for t in dst:
                assert torch.equal(t, plain)
            pD, pI = ix.search_filtered_shard(q_op, k, sel, tau, compact=compact)
            ds = [torch.full((Q, k), float("nan"), device="cuda") for _ in range(2)]
            di = [torch.full((Q, k), 7, dtype=torch.int64, device="cuda") for _ in range(2)]
            ix.search_filtered_shard(q_op, k, sel, tau, dst=([t.data_ptr() for t in ds], [t.data_ptr() for t in di]),
                                     compact=compact)
            for s_, i_ in zip(ds, di):
                assert torch.equal(s_, pD) and torch.equal(i_, pI)
            if sel.n_allowed == 0:
                assert (pI == -1).all() and (pD == -torch.finfo(torch.float32).max).all()
                assert (plain == -torch.finfo(torch.float32).max).all()
            else:
                lo, hi = ix.row_offset, ix.row_offset + ix.ntotal
                got = pI[pI >= 0].cpu().numpy()
                assert ((got >= lo) & (got < hi)).all() and mask[got].all()      # global ids of allowed rows


def test_sharded_index_host_calls_on_one_gpu():
    """ShardedFlatIndex without a process group (one shard): row_filter over global rows, search(sel=) and the host
    pipeline (search_numpy / search_stream) equal the single-index filtered search; the filtered and the unfiltered pipe
    never share a device search; fp32 storage is refused."""
    from b200rec.dist import ShardedFlatIndex
    from b200rec.retrieval import FlatIPDeviceIndex
    Q, k = 64, 50
    cat, qry, rng = _int_data(100_000, 64, Q, seed=12)
    ix = FlatIPDeviceIndex(64, storage="bf16")
    ix.add(cat)
    sh = ShardedFlatIndex.from_device_index(ix)
    rows = rng.permutation(cat.shape[0])[:3000]
    mask = np.zeros(cat.shape[0], bool)
    mask[rows] = True
    rD, rI = oracle_allowed(cat, qry, k, mask)
    uD, uI = [t.cpu().numpy() for t in ix.search_device(ix.prepare_queries(qry), k)]
    sel = sh.row_filter(rows=np.concatenate([rows, rows[:10], [-4, 10 ** 9]]))
    d, i = sh.search(ix.prepare_queries(qry), k, sel=sel)
    assert np.array_equal(i.cpu().numpy(), rI) and np.array_equal(d.cpu().numpy(), rD)
    for _ in range(2):                                                  # alternate: each call keeps its own search
        D_, I_ = sh.search_numpy(qry, k, sel=sel)
        assert np.array_equal(I_, rI) and np.array_equal(D_, rD)
        D_, I_ = sh.search_numpy(qry, k)
        assert np.array_equal(I_, uI) and np.array_equal(D_, uD)
    sel2 = sh.row_filter(mask=mask[:50_000])
    r2 = oracle_allowed(cat, qry, k, np.concatenate([mask[:50_000], np.zeros(50_000, bool)]))
    outs = list(sh.search_stream([qry[:30], qry[30:]], k, sel=sel2))
    assert np.array_equal(np.concatenate([o[1] for o in outs]), r2[1])
    f32 = FlatIPDeviceIndex(64, storage="fp32")
    f32.add(cat[:1000])
    with pytest.raises(ValueError, match="bf16"):
        ShardedFlatIndex.from_device_index(f32).row_filter(rows=[1, 2])


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
@pytest.mark.parametrize("peer", ["1", "0"])
def test_two_gpu_sharded_filtered_search_equals_single_gpu(peer):
    """Two NCCL ranks search with filters over the peer-memory path (PEER=1) and the NCCL all-gather path (PEER=0):
    tools/check_sharded_filtered.py exits non-zero unless every result is bit-identical to the single-GPU filtered
    search on the same rows."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, PEER=peer, NROWS="1000000", NQ="512")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29581" if peer == "1" else "29583",
                        os.path.join(root, "tools", "check_sharded_filtered.py")],
                       cwd=root, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
