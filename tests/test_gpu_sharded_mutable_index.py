"""GPU parity of the live catalogue on the row-sharded index: unequal row shards of one catalogue emulated on one GPU
take global-row updates and removals sliced as every rank slices them (dist.shard_update_rows / shard_filter_rows) and
run the steps every rank runs — sample_shard (live rows only, padding where a shard has nothing to sample), pooled k-th,
search_shard from that threshold, k-way merge — bit for bit against the CPU oracle over the live rows and against one
FlatIPDeviceIndex given the same mutations, on integer data with massive ties; filters built before the mutations on
every per-shard path; the unchanged launches of an index without removed rows; compact(); the host calls of
ShardedFlatIndex on one GPU; fp32 storage; and, on two GPUs, tools/check_sharded_mutable.py over both exchange
paths."""
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


def _setup(N, D, Q, seed, cat=None, qry=None, storage="bf16"):
    """(shards, single index over all rows, cat, qry, rng) on integer data (bf16-exact values, exact fp32 sums)."""
    from b200rec.retrieval import FlatIPDeviceIndex
    rng = np.random.default_rng(seed)
    if cat is None:
        cat = rng.integers(-2, 3, size=(N, D)).astype(np.float32)
        qry = rng.integers(-2, 3, size=(Q, D)).astype(np.float32)
    shards = []
    for lo, hi in SPANS:
        ix = FlatIPDeviceIndex(D, storage=storage, row_offset=lo)
        ix.add(cat[lo:hi])
        shards.append(ix)
    full = FlatIPDeviceIndex(D, storage=storage)
    full.add(cat)
    return shards, full, cat, qry, rng


def _update(shards, full, cat, live, rows, x):
    """One global update as every rank applies it, on the single index and on the CPU mirror."""
    from b200rec.dist import shard_update_rows
    for ix in shards:
        local, pos = shard_update_rows(ix.row_offset, ix.ntotal, rows)
        if local.size:
            ix.update_rows(local, x[pos])
    full.update_rows(rows, x)
    for r, v in zip(rows, x):
        cat[r] = v
    live[rows] = True


def _remove(shards, full, live, rows):
    from b200rec.dist import shard_filter_rows
    u = np.unique(rows)
    n = [ix.remove_rows(shard_filter_rows(ix.row_offset, ix.ntotal, rows=rows)) for ix in shards]
    assert sum(n) == int(live[u].sum()) == full.remove_rows(rows)
    live[rows] = False


def _random_round(shards, full, cat, live, rng, n_upd, n_rm):
    N, D = cat.shape
    rows = rng.integers(0, N, size=n_upd)
    for j, (lo, _) in enumerate(SPANS[1:]):                          # updates straddle every shard boundary
        rows[40 * j: 40 * j + 20] = lo - 10 + np.arange(20)
        rows[40 * j + 20: 40 * j + 40] = lo + 9 - np.arange(20)      # duplicates: the later value wins
    dead = np.flatnonzero(~live)[: n_upd // 5]
    rows[rows.size - dead.size:] = dead                              # revive removed rows
    _update(shards, full, cat, live, rows, rng.integers(-2, 3, size=(n_upd, D)).astype(np.float32))
    rm = rng.integers(0, N, size=n_rm)
    _remove(shards, full, live, np.concatenate([rm, rm[:5], np.flatnonzero(~live)[:5]]))


def _filters(shards, mask):
    from b200rec.dist import shard_filter_rows
    return [ix.row_filter(rows=shard_filter_rows(ix.row_offset, ix.ntotal, mask=mask)) for ix in shards]


def _sharded(shards, q_op, k, sels=None):
    """What every rank runs, with the exchange done on one device: (tau [Q] or None, D [Q,k], I [Q,k]).  Unfiltered
    shards without removed rows may have no sampling pass: then every shard agrees on no threshold."""
    from b200rec import kernels as KR
    from b200rec.dist import ShardedFlatIndex
    world = len(shards)
    sels = sels or [None] * world
    kx = ShardedFlatIndex.exchange_width(k, world)
    vals = [ix.sample_shard(q_op, k, kx, world, sel=s) for ix, s in zip(shards, sels)]
    tau = None if any(v is None for v in vals) else KR.topk_pooled_kth(torch.stack(vals).contiguous(), k)
    parts = [ix.search_shard(q_op, k, tau, sel=s) for ix, s in zip(shards, sels)]
    D, I = KR.topk_merge(torch.stack([p[0] for p in parts]).contiguous(), torch.stack([p[1] for p in parts]).contiguous(), k)
    return None if tau is None else tau.cpu().numpy(), D.cpu().numpy(), I.cpu().numpy()


def _check(shards, full, q_op, qf, cat, qry, k, mask, what, sels=None, sel_full=None):
    tau, D_, I_ = _sharded(shards, q_op, k, sels)
    rD, rI = oracle_allowed(cat, qry, k, mask)
    assert np.array_equal(I_, rI), what
    assert np.array_equal(D_, rD), what
    if tau is not None:
        assert (tau <= rD[:, k - 1]).all(), what
    fD, fI = [t.cpu().numpy() for t in full.search_device(qf, k, sel=sel_full)]
    assert np.array_equal(fI, I_) and np.array_equal(fD, D_), what
    return tau


@pytest.mark.parametrize("Q,k", [(300, 10), (300, 100), (300, 1000), (40, 10), (40, 100), (40, 1000)])
def test_random_mutations_equal_the_oracle_and_one_index(Q, k):
    """Q >= 256 runs the CTA-pair kernel, Q < 256 the single-CTA one; k = 1000 has no sampling pass on any shard, and at
    k = 10 / 100 the 40 K-row shard has none either (it pools padding)."""
    shards, full, cat, qry, rng = _setup(SPANS[-1][1], 64, Q, seed=Q + k)
    live = np.ones(cat.shape[0], bool)
    q_op, qf = shards[0].prepare_queries(qry), full.prepare_queries(qry)
    _check(shards, full, q_op, qf, cat, qry, k, live, "unmutated")
    for rnd, n_rm in enumerate((20, 2000, 30_000)):
        _random_round(shards, full, cat, live, rng, 2000, n_rm)
        _check(shards, full, q_op, qf, cat, qry, k, live, rnd)


@pytest.mark.parametrize("Q", [300, 40])
def test_pooled_threshold_ignores_removed_rows_on_every_shard(Q):
    """Every removed row outscores every live row on every shard: a shard whose sample read removed rows would pool a
    threshold above every live score and the search would return nothing."""
    N, D, k = SPANS[-1][1], 64, 100
    rng = np.random.default_rng(Q)
    dead = rng.random(N) < 0.1
    cat = -rng.integers(1, 3, size=(N, D)).astype(np.float32)
    cat[dead] = rng.integers(1, 3, size=(int(dead.sum()), D)).astype(np.float32)
    qry = rng.integers(1, 3, size=(Q, D)).astype(np.float32)
    shards, full, cat, qry, _ = _setup(N, D, Q, 0, cat, qry)
    assert all(ix.has_sample_pass(Q, k) for ix in shards[1:])
    live = np.ones(N, bool)
    _remove(shards, full, live, np.flatnonzero(dead))
    q_op, qf = shards[0].prepare_queries(qry), full.prepare_queries(qry)
    tau = _check(shards, full, q_op, qf, cat, qry, k, live, "trap")
    assert tau is not None and (tau > -3.0e38).any()                 # two sampling shards pool >= k real values


def test_a_shard_with_every_row_removed_and_fewer_than_k_live_rows_pad():
    Q, k = 300, 100
    shards, full, cat, qry, rng = _setup(SPANS[-1][1], 64, Q, seed=3)
    live = np.ones(cat.shape[0], bool)
    q_op, qf = shards[0].prepare_queries(qry), full.prepare_queries(qry)
    _remove(shards, full, live, np.arange(*SPANS[1]))                # the middle shard: nothing live
    assert shards[1].n_live == 0
    _check(shards, full, q_op, qf, cat, qry, k, live, "middle shard empty")
    keep = rng.permutation(np.flatnonzero(live))[:37]
    _remove(shards, full, live, np.setdiff1d(np.flatnonzero(live), keep))
    _check(shards, full, q_op, qf, cat, qry, k, live, "37 live rows")
    vals = shards[1].sample_shard(q_op, k, 40, 3)
    assert (vals == -torch.finfo(torch.float32).max).all()
    _update(shards, full, cat, live, np.array([SPANS[1][0] + 7, SPANS[2][0] - 1]),
            np.full((2, 64), 2.0, np.float32))                      # freed slots take new items
    _check(shards, full, q_op, qf, cat, qry, k, live, "revived")


def _path_mask(N, rng, paths):
    """A global filter whose allowed fraction on each shard selects the path in `paths` (compact below 0.75)."""
    mask = np.zeros(N, bool)
    for (lo, hi), compact in zip(SPANS, paths):
        mask[lo:hi] = rng.random(hi - lo) < (0.3 if compact else 0.9)
    return mask


@pytest.mark.parametrize("Q,k", [(300, 100), (40, 10), (40, 1000)])
def test_filters_built_before_the_mutations_on_every_path(Q, k):
    shards, full, cat, qry, rng = _setup(SPANS[-1][1], 64, Q, seed=17 + k)
    live = np.ones(cat.shape[0], bool)
    q_op, qf = shards[0].prepare_queries(qry), full.prepare_queries(qry)
    cases = []
    for paths in PATHS:
        mask = _path_mask(cat.shape[0], rng, paths)
        sels = _filters(shards, mask)
        assert [s.fraction < s.index.FILTER_COMPACT_BELOW for s in sels] == list(paths)
        _sharded(shards, q_op, k, sels)                              # gather the compacted copies before the mutations
        cases.append((paths, mask, sels, full.row_filter(mask=mask)))
    for rnd, n_rm in enumerate((500, 20_000)):
        _random_round(shards, full, cat, live, rng, 3000, n_rm)
        for paths, mask, sels, sel_full in cases:
            _check(shards, full, q_op, qf, cat, qry, k, mask & live, (rnd, paths), sels, sel_full)


def test_masked_fanout_equals_its_plain_form():
    """The new entry point on a compact shard with removed rows (compact live bits + remap together): two local
    destinations stand in for two peers' gather buffers and both receive what b200rec_flat_ip_topk_masked returns, with
    and without a threshold; and padding rows to every destination when nothing is allowed."""
    from b200rec import kernels as KR
    Q, k = 300, 100
    shards, full, cat, qry, rng = _setup(SPANS[-1][1], 64, Q, seed=5)
    live = np.ones(cat.shape[0], bool)
    q_op = shards[0].prepare_queries(qry)
    sels = _filters(shards, rng.random(cat.shape[0]) < 0.3)
    _random_round(shards, full, cat, live, rng, 2000, 20_000)
    for ix, sel in zip(shards, sels):
        cat_c = sel.compacted()
        assert sel._compact_bits is not None
        ws = ix._workspace(Q, k, cat_c.shape[0])
        for tau in (None, torch.full((Q,), 4.0, device="cuda")):
            pD, pI = KR.flat_ip_topk_masked(cat_c, q_op, k, ix.row_offset, allow_bits=sel._compact_bits,
                                             allow_n=sel.n_allowed, remap_rows=sel.rows, tau_init=tau, workspace=ws)
            ds = [torch.full((Q, k), float("nan"), device="cuda") for _ in range(2)]
            di = [torch.full((Q, k), 7, dtype=torch.int64, device="cuda") for _ in range(2)]
            KR.flat_ip_topk_masked_fanout(cat_c, q_op, k, ix.row_offset, sel._compact_bits, sel.n_allowed, sel.rows,
                                          tau, [t.data_ptr() for t in ds], [t.data_ptr() for t in di], ws)
            for s_, i_ in zip(ds, di):
                assert torch.equal(s_, pD) and torch.equal(i_, pI)
    ds = [torch.zeros((Q, k), device="cuda") for _ in range(2)]
    di = [torch.zeros((Q, k), dtype=torch.int64, device="cuda") for _ in range(2)]
    KR.flat_ip_topk_masked_fanout(None, q_op, k, 0, None, 0, None, None, [t.data_ptr() for t in ds],
                                  [t.data_ptr() for t in di], None)
    for s_, i_ in zip(ds, di):
        assert (i_ == -1).all() and (s_ == -torch.finfo(torch.float32).max).all()


def _launches(fn):
    from b200rec import _native
    torch.cuda.synchronize()
    before = _native.launch_count()
    out = fn()
    torch.cuda.synchronize()
    return out, _native.launch_count() - before


def _bytes(out):
    if out is None:
        return None
    if torch.is_tensor(out):
        return out.cpu().numpy().tobytes()
    return tuple(t.cpu().numpy().tobytes() for t in out)


@pytest.mark.parametrize("updated", [False, True])
def test_without_removed_rows_the_new_steps_run_the_old_launches(updated):
    """An unmutated index, and one that took updates alone, run exactly the launches of sample_device / sample_fanout /
    search_device(tau_init=) / search_fanout / sample_filtered / search_filtered_shard and return the same bytes."""
    Q, k = 300, 100
    shards, full, cat, qry, rng = _setup(SPANS[-1][1], 64, Q, seed=23)
    live = np.ones(cat.shape[0], bool)
    if updated:
        rows = rng.integers(0, cat.shape[0], size=20_000)
        _update(shards, full, cat, live, rows, rng.integers(-2, 3, size=(rows.size, 64)).astype(np.float32))
    ix = shards[2]
    assert ix._live_bits is None and ix.has_sample_pass(Q, k)
    q_op = ix.prepare_queries(qry)
    tau = torch.full((Q,), 3.0, device="cuda")
    sels = {c: ix.row_filter(mask=rng.random(ix.ntotal) < (0.3 if c else 0.9)) for c in (False, True)}

    def dst(shape, dtype=torch.float32):
        ts = [torch.zeros(shape, dtype=dtype, device="cuda") for _ in range(2)]
        return ts, [t.data_ptr() for t in ts]
    pairs = [(lambda: ix.sample_device(q_op, k, 40, 3), lambda: ix.sample_shard(q_op, k, 40, 3)),
             (lambda: ix.search_device(q_op, k, tau_init=tau), lambda: ix.search_shard(q_op, k, tau))]
    for c, sel in sels.items():
        pairs += [(lambda sel=sel: ix.sample_filtered(q_op, k, 40, 3, sel), lambda sel=sel: ix.sample_shard(q_op, k, 40, 3, sel=sel)),
                  (lambda sel=sel: ix.search_filtered_shard(q_op, k, sel, tau), lambda sel=sel: ix.search_shard(q_op, k, tau, sel=sel))]
    for old, new in pairs:
        old()                                                        # a compact filter gathers its rows on first use
        a, na = _launches(old)
        b, nb = _launches(new)
        assert na == nb and _bytes(a) == _bytes(b)
    for sel in (None, sels[False], sels[True]):                       # the fan-out forms
        (va, pa), (vb, pb) = dst((Q, 40)), dst((Q, 40))
        old = (lambda: ix.sample_fanout(q_op, k, 40, 3, pa)) if sel is None else \
            (lambda: ix.sample_filtered(q_op, k, 40, 3, sel, dst=pa))
        _, na = _launches(old)
        _, nb = _launches(lambda: ix.sample_shard(q_op, k, 40, 3, sel=sel, dst=pb))
        assert na == nb and all(torch.equal(x, y) for x, y in zip(va, vb))
        (sa, psa), (ia, pia) = dst((Q, k)), dst((Q, k), torch.int64)
        (sb, psb), (ib, pib) = dst((Q, k)), dst((Q, k), torch.int64)
        old = (lambda: ix.search_fanout(q_op, k, tau, psa, pia)) if sel is None else \
            (lambda: ix.search_filtered_shard(q_op, k, sel, tau, dst=(psa, pia)))
        _, na = _launches(old)
        _, nb = _launches(lambda: ix.search_shard(q_op, k, tau, sel=sel, dst=(psb, pib)))
        assert na == nb and all(torch.equal(x, y) for x, y in zip(sa + ia, sb + ib))


def test_compact_keeps_the_results_moves_the_offsets_and_rejects_old_filters():
    """Each shard compacts, the offsets become the prefix sums of the new shard sizes, and the results mapped through
    the global old -> new map equal the results before.  The last shard keeps too few rows for a sampling pass at this
    shape, so afterwards it pools nothing (the emulated agreement drops the threshold) and results are unchanged."""
    from b200rec.dist import ShardedFlatIndex
    Q, k = 300, 100
    shards, full, cat, qry, rng = _setup(SPANS[-1][1], 64, Q, seed=29)
    live = np.ones(cat.shape[0], bool)
    q_op = shards[0].prepare_queries(qry)
    _random_round(shards, full, cat, live, rng, 2000, 30_000)
    _remove(shards, full, live, np.arange(SPANS[2][0] + 1000, SPANS[2][1]))   # the last shard keeps < 1000 rows
    assert shards[2].has_sample_pass(Q, k)
    mask = _path_mask(cat.shape[0], rng, PATHS[2])
    sels = _filters(shards, mask)
    _, bD, bI = _sharded(shards, q_op, k)
    _, fD, fI = _sharded(shards, q_op, k, sels)
    remap = np.full(cat.shape[0], -1, np.int64)
    off = 0
    for ix in shards:
        old = ix.row_offset
        local = ix.compact()
        kept = local >= 0
        remap[old + np.flatnonzero(kept)] = off + local[kept]
        ix.row_offset = off
        off += ix.ntotal
    assert shards[1].row_offset < SPANS[1][0] and not shards[2].has_sample_pass(Q, k)
    assert np.array_equal(remap[live], np.arange(int(live.sum())))
    _, aD, aI = _sharded(shards, q_op, k)
    assert np.array_equal(aD, bD) and np.array_equal(aI, np.where(bI >= 0, remap[np.maximum(bI, 0)], -1))
    _, gD, gI = _sharded(shards, q_op, k, _filters(shards, mask[live]))
    assert np.array_equal(gD, fD) and np.array_equal(gI, np.where(fI >= 0, remap[np.maximum(fI, 0)], -1))
    for ix, sel in zip(shards, sels):
        with pytest.raises(ValueError, match="compact"):
            ix.search_shard(q_op, k, None, sel=sel)
        with pytest.raises(ValueError, match="compact"):
            ix.sample_shard(q_op, k, 40, 3, sel=sel)
    sh = ShardedFlatIndex.from_device_index(shards[0])                 # no process group: one shard
    sh._ids_cache[("use", Q, k)] = True
    sh._ids_cache[("peer", Q, k)] = None
    sh.compact()
    assert not any(key[0] in ("use", "peer") for key in sh._ids_cache)


def test_sharded_index_host_calls_on_one_gpu():
    """ShardedFlatIndex without a process group passes the mutation calls through to its index: search, search(sel=),
    search_numpy and a search_stream batch submitted after an update see the update; n_live and compact() agree with the
    index; an fp32-storage shard with removed rows refuses the row-shard steps."""
    from b200rec.dist import ShardedFlatIndex
    from b200rec.retrieval import FlatIPDeviceIndex
    N, D, Q, k = 100_000, 64, 64, 50
    rng = np.random.default_rng(31)
    cat = rng.integers(-2, 3, size=(N, D)).astype(np.float32)
    qry = rng.integers(-2, 3, size=(Q, D)).astype(np.float32)
    ix = FlatIPDeviceIndex(D, storage="bf16")
    ix.add(cat)
    sh = ShardedFlatIndex.from_device_index(ix)
    live = np.ones(N, bool)
    mask = rng.random(N) < 0.3
    sel = sh.row_filter(mask=mask)
    rows = rng.permutation(N)[:500]
    x = np.full((rows.size, D), 2.0, np.float32)                      # the new rows outscore many old ones
    before = cat.copy()

    def batches():
        yield qry
        sh.update_rows(rows, x)
        assert sh.remove_rows(rows[:100]) == 100
        yield qry
    first, second = list(sh.search_stream(batches(), k))
    cat[rows] = x
    live[rows[:100]] = False
    for got, xb, m in ((first, before, np.ones(N, bool)), (second, cat, live)):
        rD, rI = oracle_allowed(xb, qry, k, m)
        assert np.array_equal(got[1], rI) and np.array_equal(got[0], rD)
    assert sh.n_live() == ix.n_live == N - 100
    rD, rI = oracle_allowed(cat, qry, k, mask & live)
    for got in (sh.search_numpy(qry, k, sel=sel), [t.cpu().numpy() for t in sh.search(ix.prepare_queries(qry), k, sel=sel)]):
        assert np.array_equal(got[1], rI) and np.array_equal(got[0], rD)
    remap = sh.compact()
    assert np.array_equal(remap, np.where(live, np.cumsum(live) - 1, -1)) and sh.n_live() == ix.ntotal
    f32 = FlatIPDeviceIndex(D, storage="fp32")
    f32.add(cat[:5000])
    f32.remove_rows([3])
    q32 = f32.prepare_queries(qry)
    with pytest.raises(ValueError, match="bf16"):
        f32.search_shard(q32, k, None)
    with pytest.raises(ValueError, match="bf16"):
        f32.sample_shard(q32, k, 20, 2)
    d32, i32 = ShardedFlatIndex.from_device_index(f32).search(q32, k)   # one GPU: the single-index search, any storage
    assert not (i32 == 3).any()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
@pytest.mark.parametrize("peer", ["1", "0"])
def test_two_gpu_sharded_mutable_search_equals_single_gpu(peer):
    """Two NCCL ranks mutate and search over the peer-memory path (PEER=1) and the NCCL all-gather path (PEER=0):
    tools/check_sharded_mutable.py exits non-zero unless every result is bit-identical to the single-GPU search over the
    same mutated rows."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, PEER=peer, NROWS="1000000", NQ="512")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29585" if peer == "1" else "29587",
                        os.path.join(root, "tools", "check_sharded_mutable.py")],
                       cwd=root, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
