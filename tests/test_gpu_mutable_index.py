"""GPU parity of the mutable catalogue (FlatIPDeviceIndex.update_rows / remove_rows / compact and B200FlatIndex's
"updates": "in_place"): every search path returns the exact top-k over the LIVE rows with their current contents, bit for
bit against the CPU oracle over a mirror of the rows and the live mask (`oracle_allowed`), on integer data with massive
ties; the sampling-pass trap with removed rows; padding; the unchanged fast path after updates alone; row filters built
before the mutations (bitmap and compact paths, the cached compact copy patched in place); exclusion lists; fp32
storage; the faiss normalisation rule; compact(); search_stream ordering; the guarded row-shard entry points; the
drop-in engine under a Kafka-like stream of upserts and removals."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


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


def _int_index(N, D, Q, seed, storage="bf16"):
    from b200rec.retrieval import FlatIPDeviceIndex
    rng = np.random.default_rng(seed)
    cat = rng.integers(-2, 3, size=(N, D)).astype(np.float32)         # bf16-exact values, exact fp32 sums: massive ties
    qry = rng.integers(-2, 3, size=(Q, D)).astype(np.float32)
    ix = FlatIPDeviceIndex(D, storage=storage)
    ix.add(cat)
    return ix, cat, qry, rng


def _host(t):
    return [x.cpu().numpy() for x in t]


def _assert_oracle(got, cat, qry, k, mask, what=""):
    rD, rI = oracle_allowed(cat, qry, k, mask)
    D_, I_ = got
    assert np.array_equal(I_, rI), what
    assert np.array_equal(D_, rD), what


def _mutate(ix, cat, live, rng, n_upd, n_rm, D):
    """One random batch of each kind on the device index and on the CPU mirror: updates with duplicate rows (the last
    occurrence wins; some hit removed rows and revive them), removals with duplicates and already-removed rows."""
    rows = rng.integers(0, ix.ntotal, size=n_upd)
    rows[: n_upd // 10] = rows[n_upd // 10: 2 * (n_upd // 10)]                      # duplicates inside the batch
    dead = np.flatnonzero(~live)
    if dead.size:
        rows[-min(dead.size, n_upd // 5):] = dead[: min(dead.size, n_upd // 5)]     # revive removed rows
    x = rng.integers(-2, 3, size=(n_upd, D)).astype(np.float32)
    ix.update_rows(rows, x)
    for r, v in zip(rows, x):
        cat[r] = v
    live[rows] = True
    rm = rng.integers(0, ix.ntotal, size=n_rm)
    rm = np.concatenate([rm, rm[:5], np.flatnonzero(~live)[:5]])
    was = int(np.count_nonzero(live[np.unique(rm)]))
    assert ix.remove_rows(rm) == was
    live[rm] = False
    assert ix.n_live == int(live.sum())


@pytest.mark.parametrize("Q,k", [(300, 10), (300, 100), (40, 100), (40, 1000)])
def test_random_mutation_sequences_equal_the_oracle_over_live_rows(Q, k):
    """Q >= 256 runs the CTA-pair kernel, Q < 256 the single-CTA one; k = 10 / 100 run the masked sampling pass,
    k = 1000 does not.  Interleaved update / remove / revive / add rounds, both search entry points."""
    N, D = 200_000, 64
    ix, cat, qry, rng = _int_index(N, D, Q, seed=Q + k)
    live = np.ones(N, bool)
    q_op = ix.prepare_queries(qry)
    for rnd in range(4):
        _mutate(ix, cat, live, rng, n_upd=2000, n_rm=(20, 2000, 30_000, 100)[rnd], D=D)
        if rnd == 2:                                                        # appended rows are live
            extra = rng.integers(-2, 3, size=(5000, D)).astype(np.float32)
            ix.add(extra)
            cat = np.concatenate([cat, extra])
            live = np.concatenate([live, np.ones(len(extra), bool)])
        _assert_oracle(_host(ix.search_device(q_op, k)), cat, qry, k, live, rnd)
    _assert_oracle(ix.search(qry, k), cat, qry, k, live, "host")


@pytest.mark.parametrize("Q", [300, 40])
def test_sampling_threshold_ignores_removed_rows(Q):
    """Every removed row outscores every live row for every query: a threshold seeded from them would return nothing."""
    from b200rec.retrieval import FlatIPDeviceIndex
    N, D, k = 200_000, 64, 100
    rng = np.random.default_rng(Q)
    dead = rng.permutation(N)[: N // 10]
    cat = -rng.integers(1, 3, size=(N, D)).astype(np.float32)
    cat[dead] = rng.integers(1, 3, size=(dead.size, D)).astype(np.float32)
    qry = rng.integers(1, 3, size=(Q, D)).astype(np.float32)
    ix = FlatIPDeviceIndex(D, storage="bf16")
    ix.add(cat)
    ix.remove_rows(dead)
    assert ix.has_sample_pass(Q, k)
    live = np.ones(N, bool)
    live[dead] = False
    rD, _ = oracle_allowed(cat, qry, k, live)
    assert (rD < 0).all()
    _assert_oracle(_host(ix.search_device(ix.prepare_queries(qry), k)), cat, qry, k, live)


def test_fewer_than_k_live_rows_and_all_rows_removed_pad():
    N, D, Q, k = 5000, 64, 8, 100
    ix, cat, qry, rng = _int_index(N, D, Q, seed=2)
    live = np.zeros(N, bool)
    keep = rng.permutation(N)[:37]
    live[keep] = True
    assert ix.remove_rows(np.flatnonzero(~live)) == N - 37
    q_op = ix.prepare_queries(qry)
    _assert_oracle(_host(ix.search_device(q_op, k)), cat, qry, k, live)
    assert ix.remove_rows(keep) == 37 and ix.n_live == 0
    D_, I_ = _host(ix.search_device(q_op, k))
    assert (I_ == -1).all() and (D_ == -np.finfo(np.float32).max).all()
    assert (ix.search(qry, k)[1] == -1).all()


def test_updates_alone_keep_the_fast_path_and_equal_a_fresh_index():
    from b200rec import _native
    from b200rec.retrieval import FlatIPDeviceIndex
    N, D, Q, k = 200_000, 64, 300, 100
    ix, cat, qry, rng = _int_index(N, D, Q, seed=5)
    rows = rng.integers(0, N, size=20_000)
    x = rng.integers(-2, 3, size=(rows.size, D)).astype(np.float32)
    ix.update_rows(rows, x)
    for r, v in zip(rows, x):
        cat[r] = v
    assert ix._live_bits is None and ix.n_live == N                   # no removal: no live bitmap, unchanged path
    fresh = FlatIPDeviceIndex(D, storage="bf16")
    fresh.add(cat)
    got = []
    for index in (ix, fresh):
        q_op = index.prepare_queries(qry)
        torch.cuda.synchronize()
        before = _native.launch_count()
        got.append(_host(index.search_device(q_op, k)))
        torch.cuda.synchronize()
        got[-1].append(_native.launch_count() - before)
    assert got[0][0].tobytes() == got[1][0].tobytes() and got[0][1].tobytes() == got[1][1].tobytes()
    assert got[0][2] == got[1][2]
    assert torch.equal(ix._cat[:N], fresh._cat[:N])


@pytest.mark.parametrize("Q,k", [(300, 100), (40, 1000)])
def test_filters_built_before_mutations_answer_over_filter_and_live_rows(Q, k):
    N, D = 200_000, 64
    ix, cat, qry, rng = _int_index(N, D, Q, seed=7 + k)
    mask = rng.random(N) < 0.3
    sel = ix.row_filter(mask=mask)
    q_op = ix.prepare_queries(qry)
    _host(ix._search_filtered(q_op, k, sel, compact=True))                  # gather the compacted copy now
    cached = sel._compact
    live = np.ones(N, bool)
    for rnd in range(3):
        _mutate(ix, cat, live, rng, n_upd=3000, n_rm=(500, 20_000, 50)[rnd], D=D)
        for compact in (False, True):
            _assert_oracle(_host(ix._search_filtered(q_op, k, sel, compact)), cat, qry, k, mask & live, (rnd, compact))
        _assert_oracle(ix.search(qry, k, sel=sel), cat, qry, k, mask & live, "selected path")
    assert sel._compact is cached                                            # patched in place, never re-gathered
    fresh = ix.row_filter(mask=mask)
    assert torch.equal(fresh.compacted(), cached)
    for compact in (False, True):
        a = _host(ix._search_filtered(q_op, k, fresh, compact))
        _assert_oracle(a, cat, qry, k, mask & live, ("fresh", compact))


def test_exclusion_lists_on_an_index_with_removed_rows():
    from b200rec.retrieval import exact_topk_eval
    from oracle.flat_ip import IndexFlatIP
    N, D, Q, k = 100_000, 64, 50, 100
    ix, cat, qry, rng = _int_index(N, D, Q, seed=9)
    dead = rng.permutation(N)[:15_000]
    ix.remove_rows(dead)
    train = {u: rng.integers(0, N, size=int(rng.integers(0, 300))).tolist() for u in range(Q)}
    ids = exact_topk_eval(torch.from_numpy(qry).cuda(), ix, train, list(range(Q)), k)
    ref = IndexFlatIP(D)
    ref.add(cat)
    _, rI = ref.search(qry, k, exclude=[np.union1d(np.asarray(train[u], np.int64), dead) for u in range(Q)])
    assert np.array_equal(ids, rI)


@pytest.mark.parametrize("D", [128, 100])
def test_fp32_storage_after_updates_matches_the_fp32_oracle(D):
    """Tolerances of test_fp32_storage_with_a_filter_matches_the_fp32_oracle: scores within 1e-6, ids equal except inside
    scores tied within 1e-6 (fp32 summation order)."""
    from b200rec.retrieval import FlatIPDeviceIndex
    from oracle.flat_ip import normalize_L2
    rng = np.random.default_rng(D)
    N, Q, k = 20000, 70, 100
    cat = normalize_L2(rng.standard_normal((N, D)).astype(np.float32))
    qry = normalize_L2(rng.standard_normal((Q, D)).astype(np.float32))
    ix = FlatIPDeviceIndex(D, storage="fp32")
    ix.add(cat)
    rows = rng.permutation(N)[:3000]
    x = rng.standard_normal((rows.size, D)).astype(np.float32)
    ix.update_rows(rows, x, normalize=True)
    cat[rows] = normalize_L2(x.copy())
    live = np.ones(N, bool)
    dead = rng.permutation(N)[:4000]
    ix.remove_rows(dead)
    live[dead] = False
    q_op = ix.prepare_queries(qry)
    sel = ix.row_filter(mask=rng.random(N) < 0.3)
    mask = np.zeros(N, bool)
    mask[sel.rows.cpu().numpy()] = True
    cases = [(_host(ix.search_device(q_op, k)), live)]
    cases += [(_host(ix._search_filtered(q_op, k, sel, c)), live & mask) for c in (False, True)]
    for (Dg, Ig), m in cases:
        rD, rI = oracle_allowed(cat, qry, k, m)
        assert np.abs(Dg - rD).max() <= 1e-6
        bad = np.argwhere(Ig != rI)
        for q, j in bad:
            assert m[Ig[q, j]]
            exact = float(cat[Ig[q, j]].astype(np.float64) @ qry[q].astype(np.float64))
            assert abs(exact - rD[q, j]) <= 1e-6
        assert len(bad) <= 0.002 * Ig.size


def test_update_rows_normalize_applies_the_faiss_rule():
    from b200rec.retrieval import FlatIPDeviceIndex
    from oracle.flat_ip import normalize_L2
    rng = np.random.default_rng(1)
    D = 96
    ix = FlatIPDeviceIndex(D, storage="fp32")
    ix.add(rng.standard_normal((1000, D)).astype(np.float32), normalize=True)
    x = rng.standard_normal((6, D)).astype(np.float32)
    x[[1, 4]] = 0.0
    rows = np.array([3, 500, 999, 0, 7, 8])
    ix.update_rows(rows, x, normalize=True)
    got = ix.reconstruct_n(0, 1000)[rows]
    assert (got[[1, 4]] == 0).all()
    assert np.allclose(got, normalize_L2(x.copy()), rtol=0, atol=1e-6)


def test_compact_keeps_the_results_and_rejects_stale_filters():
    N, D, Q, k = 100_000, 64, 300, 100
    ix, cat, qry, rng = _int_index(N, D, Q, seed=11)
    live = np.ones(N, bool)
    _mutate(ix, cat, live, rng, n_upd=2000, n_rm=30_000, D=D)
    sel = ix.row_filter(mask=rng.random(N) < 0.2)
    q_op = ix.prepare_queries(qry)
    bD, bI = _host(ix.search_device(q_op, k))
    remap = ix.compact()
    assert ix.ntotal == ix.n_live == int(live.sum()) and (remap[~live] == -1).all()
    assert np.array_equal(remap[live], np.arange(int(live.sum())))
    aD, aI = _host(ix.search_device(ix.prepare_queries(qry), k))
    assert np.array_equal(aD, bD) and np.array_equal(aI, np.where(bI >= 0, remap[np.maximum(bI, 0)], -1))
    _assert_oracle((aD, aI), cat[live], qry, k, np.ones(int(live.sum()), bool))
    with pytest.raises(ValueError, match="compact"):
        ix.search_device(q_op, k, sel=sel)


def test_search_stream_batches_submitted_after_an_update_see_it():
    N, D, Q, k = 50_000, 64, 64, 20
    ix, cat, qry, rng = _int_index(N, D, Q, seed=13)
    before = cat.copy()
    rows = rng.permutation(N)[:500]
    x = np.full((rows.size, D), 2.0, np.float32)                         # the new rows outscore many old ones

    def batches():
        yield qry
        ix.update_rows(rows, x)
        ix.remove_rows(rows[:100])
        yield qry
    first, second = list(ix.search_stream(batches(), k))
    _assert_oracle(first, before, qry, k, np.ones(N, bool))
    cat[rows] = x
    live = np.ones(N, bool)
    live[rows[:100]] = False
    _assert_oracle(second, cat, qry, k, live)


def test_row_shard_entry_points_refuse_an_index_with_removed_rows():
    ix, _, qry, _ = _int_index(100_000, 64, 300, seed=3)
    sel = ix.row_filter(rows=np.arange(1000))
    q_op = ix.prepare_queries(qry)
    ix.remove_rows([5])
    calls = [lambda: ix.sample_device(q_op, 100), lambda: ix.sample_fanout(q_op, 100, 100, 2, []),
             lambda: ix.search_fanout(q_op, 100, None, [], []),
             lambda: ix.sample_filtered(q_op, 100, 100, 2, sel),
             lambda: ix.search_filtered_shard(q_op, 100, sel, None)]
    for call in calls:
        with pytest.raises(ValueError, match="removed rows"):
            call()
    ix.update_rows([5], np.zeros((1, 64), np.float32))                   # revived: the shard steps run again
    d, i = ix.search_filtered_shard(q_op, 100, sel, None)
    assert d.shape == i.shape == (300, 100)


def test_engine_in_place_updates_through_a_kafka_like_stream(tmp_path):
    from b200rec.retrieval import RetrievalEngine
    from oracle.flat_ip import normalize_L2
    rng = np.random.default_rng(21)
    N, D, k = 20_000, 64, 50
    cfg = {"index_type": "b200", "embedding_dim": D, "b200": {"metric": "cosine", "updates": "in_place"}}
    eng = RetrievalEngine(cfg)
    names = [f"item_{i}" for i in range(N)]
    emb = {n: v for n, v in zip(names, rng.standard_normal((N, D)).astype(np.float32))}
    eng.build_index(np.stack([emb[n] for n in names]), names)
    qry = rng.standard_normal((16, D)).astype(np.float32)
    sizes = []
    for step in range(20):
        ids = [names[j] for j in rng.integers(0, N, size=200)] + [f"new_{step}_{j}" for j in range(20)]
        vecs = rng.standard_normal((len(ids), D)).astype(np.float32)
        eng.update_index(vecs, ids)
        for n, v in zip(ids, vecs):
            emb[n] = v
        gone = [f"new_{step - 1}_{j}" for j in range(20)] + [names[j] for j in rng.integers(0, N, size=10)]
        eng.index.remove(gone)
        for n in gone:
            emb.pop(n, None)
        out, scores, _ = eng.retrieve(qry, k=k)
        assert all(len(set(r)) == len(r) == k for r in out)
        sizes.append(eng.index.index.ntotal)
        assert eng.get_metrics()["index_size"] == len(emb) == eng.index.index.n_live
    assert sizes[-1] == sizes[5]                                         # removed slots are reused
    live_names = sorted(emb)
    xb = normalize_L2(np.stack([emb[n] for n in live_names]))
    _, rI = oracle_allowed(xb, normalize_L2(qry.copy()), k, np.ones(len(live_names), bool))
    want = [[live_names[i] for i in r] for r in rI]
    out, _, _ = eng.retrieve(qry, k=k)
    agree = np.mean([a == b for ra, rb in zip(out, want) for a, b in zip(ra, rb)])
    assert agree >= 0.99                                                 # fp32 storage: ids differ only inside fp32 ties
    eng.save(str(tmp_path / "eng"))
    eng2 = RetrievalEngine(cfg)
    eng2.load(str(tmp_path / "eng"))
    assert eng2.index.current_size == len(emb) == eng2.index.index.ntotal
    assert eng2.retrieve(qry, k=k)[0] == out
