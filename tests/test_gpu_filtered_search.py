"""GPU parity of filtered exact search (FlatIPDeviceIndex.row_filter / sel=): both execution paths — the row bitmap
tested inside the fused kernel, and the compacted catalogue with ids mapped back — against the CPU oracle searching the
allowed rows alone (`oracle_allowed`, pinned to a brute-force lexsort in test_filtered_search_host.py), bit for bit on
integer data with massive ties; the sampling-pass threshold under a filter; fp32 storage; filter
reuse across `add`; B200FlatIndex's "filter": "exact" mode through RetrievalEngine."""
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


def _int_index(N, D, Q, seed, lo=-2, hi=3):
    from b200rec.retrieval import FlatIPDeviceIndex
    rng = np.random.default_rng(seed)
    cat = rng.integers(lo, hi, size=(N, D)).astype(np.float32)        # bf16-exact values, exact fp32 sums: massive ties
    qry = rng.integers(lo, hi, size=(Q, D)).astype(np.float32)
    ix = FlatIPDeviceIndex(D, storage="bf16")
    ix.add(cat)
    return ix, cat, qry, rng


def _both_paths(ix, q_op, k, sel):
    a = [t.cpu().numpy() for t in ix._search_filtered(q_op, k, sel, compact=False)]
    b = [t.cpu().numpy() for t in ix._search_filtered(q_op, k, sel, compact=True)]
    return a, b


@pytest.mark.parametrize("Q,k", [(300, 10), (300, 100), (40, 100), (40, 1000)])
def test_both_paths_equal_the_oracle_bit_for_bit(Q, k):
    """Q >= 256 runs the CTA-pair kernel (stream_scores2_kernel), Q < 256 the single-CTA one; k = 10 / 100 run the
    masked sampling pass, k = 1000 does not.  Allowed sets: empty, 1 row, k - 1 rows, 0.1 %, 10 %, 50 %, 100 %."""
    N, D = 200_000, 64
    ix, cat, qry, rng = _int_index(N, D, Q, seed=Q + k)
    q_op = ix.prepare_queries(qry)
    for n_allowed in (0, 1, k - 1, N // 1000, N // 10, N // 2, N):
        mask = np.zeros(N, bool)
        mask[rng.permutation(N)[:n_allowed]] = True
        sel = ix.row_filter(mask=mask)
        assert sel.n_allowed == n_allowed
        rD, rI = oracle_allowed(cat, qry, k, mask)
        (aD, aI), (bD, bI) = _both_paths(ix, q_op, k, sel)
        for D_, I_ in ((aD, aI), (bD, bI)):
            assert np.array_equal(I_, rI), n_allowed
            assert np.array_equal(D_, rD), n_allowed
        assert aD.tobytes() == bD.tobytes() and aI.tobytes() == bI.tobytes()


@pytest.mark.parametrize("Q", [300, 40])
def test_sampling_threshold_respects_the_filter(Q):
    """Every allowed row scores below every disallowed row for every query: a sampling pass that ignored the filter
    would start tau above every allowed score and return nothing.  The bitmap path must still equal the oracle."""
    from b200rec.retrieval import FlatIPDeviceIndex
    N, D, k = 200_000, 64, 100
    rng = np.random.default_rng(Q)
    mask = np.zeros(N, bool)
    mask[rng.permutation(N)[: N // 10]] = True
    cat = rng.integers(1, 3, size=(N, D)).astype(np.float32)
    cat[mask] = -rng.integers(1, 3, size=(int(mask.sum()), D)).astype(np.float32)
    qry = rng.integers(1, 3, size=(Q, D)).astype(np.float32)
    ix = FlatIPDeviceIndex(D, storage="bf16")
    ix.add(cat)
    assert ix.has_sample_pass(Q, k)
    rD, rI = oracle_allowed(cat, qry, k, mask)
    assert (rD < 0).all() and (rI >= 0).all()
    d, i = ix._search_filtered(ix.prepare_queries(qry), k, ix.row_filter(mask=mask), compact=False)
    assert np.array_equal(i.cpu().numpy(), rI) and np.array_equal(d.cpu().numpy(), rD)


def test_all_allowed_filter_equals_the_unfiltered_search():
    from b200rec.retrieval import FlatIPDeviceIndex
    rng = np.random.default_rng(9)
    N, D, Q, k = 200_000, 128, 300, 100
    ix = FlatIPDeviceIndex(D, storage="bf16")
    ix.add(rng.standard_normal((N, D)).astype(np.float32), normalize=True)
    q_op = ix.prepare_queries(rng.standard_normal((Q, D)).astype(np.float32), normalize=True)
    uD, uI = [t.cpu().numpy() for t in ix.search_device(q_op, k)]
    sel = ix.row_filter(rows=torch.arange(N))
    assert sel.fraction == 1.0
    for D_, I_ in _both_paths(ix, q_op, k, sel):
        assert D_.tobytes() == uD.tobytes() and I_.tobytes() == uI.tobytes()
    D_, I_ = [t.cpu().numpy() for t in ix.search_device(q_op, k, sel=sel)]                 # the selected path
    assert D_.tobytes() == uD.tobytes() and I_.tobytes() == uI.tobytes()


@pytest.mark.parametrize("D", [128, 100])
def test_fp32_storage_with_a_filter_matches_the_fp32_oracle(D):
    """Tolerances of test_fp32_storage_matches_the_fp32_oracle: scores within 1e-6, ids equal except inside scores tied
    within 1e-6 (fp32 summation order)."""
    from b200rec.retrieval import FlatIPDeviceIndex
    from oracle.flat_ip import normalize_L2
    rng = np.random.default_rng(D)
    N, Q, k = 20000, 70, 100
    cat = normalize_L2(rng.standard_normal((N, D)).astype(np.float32))
    qry = normalize_L2(rng.standard_normal((Q, D)).astype(np.float32))
    ix = FlatIPDeviceIndex(D, storage="fp32")
    ix.add(cat)
    for frac in (0.003, 0.3):
        mask = rng.random(N) < frac
        rD, rI = oracle_allowed(cat, qry, k, mask)
        sel = ix.row_filter(mask=mask)
        q_op = ix.prepare_queries(qry)
        for compact in (False, True):
            Dg, Ig = [t.cpu().numpy() for t in ix._search_filtered(q_op, k, sel, compact)]
            assert np.abs(Dg - rD).max() <= 1e-6
            bad = np.argwhere(Ig != rI)
            for q, j in bad:
                assert mask[Ig[q, j]]
                exact = float(cat[Ig[q, j]].astype(np.float64) @ qry[q].astype(np.float64))
                assert abs(exact - rD[q, j]) <= 1e-6
            assert len(bad) <= 0.002 * Ig.size
        Dh, Ih = ix.search(qry, k, sel=sel)                                                   # host entry point
        assert np.abs(Dh - rD).max() <= 1e-6 and (Ih == rI).mean() >= 0.998


def test_filter_reuse_and_rows_added_later():
    N, D, Q, k = 50_000, 64, 40, 50
    ix, cat, qry, rng = _int_index(N, D, Q, seed=77)
    mask = rng.random(N) < 0.01
    sel = ix.row_filter(rows=np.concatenate([np.flatnonzero(mask), np.flatnonzero(mask)[:5], [-3, N, N + 7]]))
    assert sel.n_allowed == int(mask.sum())                       # duplicates and out-of-range rows are ignored
    q_op = ix.prepare_queries(qry)
    first = [t.cpu().numpy() for t in ix._search_filtered(q_op, k, sel, compact=True)]
    cached = sel._compact
    again = [t.cpu().numpy() for t in ix._search_filtered(q_op, k, sel, compact=True)]
    assert sel._compact is cached
    assert all(a.tobytes() == b.tobytes() for a, b in zip(first, again))
    extra = rng.integers(-2, 3, size=(3000, D)).astype(np.float32) + 3               # would outscore every old row
    ix.add(extra)
    rD, rI = oracle_allowed(np.concatenate([cat, extra]), qry, k, np.concatenate([mask, np.zeros(len(extra), bool)]))
    for compact in (False, True):
        D_, I_ = [t.cpu().numpy() for t in ix._search_filtered(ix.prepare_queries(qry), k, sel, compact)]
        assert np.array_equal(I_, rI) and np.array_equal(D_, rD)


@pytest.mark.parametrize("metric", ["cosine", "ip"])
def test_exact_filter_mode_through_the_retrieval_engine(metric):
    from b200rec.retrieval import RetrievalEngine
    from oracle.flat_ip import normalize_L2
    rng = np.random.default_rng(4)
    N, D, k = 3000, 32, 10
    emb = rng.standard_normal((N, D)).astype(np.float32)
    qry = rng.standard_normal((6, D)).astype(np.float32)
    names = [f"item_{i}" for i in range(N)]
    eng = RetrievalEngine({"index_type": "b200", "embedding_dim": D, "b200": {"metric": metric, "filter": "exact"}})
    eng.build_index(emb.copy(), names)
    xb = normalize_L2(emb.copy()) if metric == "cosine" else emb
    q = normalize_L2(qry.copy()) if metric == "cosine" else qry
    for n_allowed in (4, 30, 600):
        rows = rng.permutation(N)[:n_allowed]
        fids = [names[r] for r in rows] + ["not_an_item"]
        ids, scores, m = eng.retrieve(qry.copy(), k=k, filter_ids=fids)
        mask = np.zeros(N, bool)
        mask[rows] = True
        _, rI = oracle_allowed(xb, q, k, mask)
        assert ids == [[names[i] for i in r if i >= 0] for r in rI]
        assert all(len(r) == min(k, n_allowed) and set(r) <= set(fids) for r in ids)
        assert m["num_results"] == 6 * min(k, n_allowed)
    assert eng.retrieve(qry.copy(), k=k, filter_ids=[])[0] == [[]] * 6


def test_filter_rejects_exclusion_lists_and_tau_init():
    from b200rec.retrieval import FlatIPDeviceIndex
    ix, _, qry, _ = _int_index(5000, 64, 8, seed=1)
    sel = ix.row_filter(rows=[1, 2, 3])
    q_op = ix.prepare_queries(qry)
    indptr = torch.zeros(9, dtype=torch.int64, device="cuda")
    rows = torch.zeros(1, dtype=torch.int32, device="cuda")
    with pytest.raises(ValueError, match="exclusion"):
        ix.search_device(q_op, 5, indptr, rows, sel=sel)
    with pytest.raises(ValueError, match="tau_init"):
        ix.search_device(q_op, 5, tau_init=torch.zeros(8, device="cuda"), sel=sel)
    other = FlatIPDeviceIndex(64, storage="bf16")
    other.add(np.zeros((10, 64), np.float32))
    with pytest.raises(ValueError, match="another index"):
        other.search_device(other.prepare_queries(qry), 5, sel=sel)
