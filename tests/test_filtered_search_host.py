"""CPU checks of filtered exact search (no GPU): the filtered reference search the GPU tests compare with (the oracle over
the allowed rows only, ids mapped back) against a brute-force lexsort and against the oracle's exclusion masking of the
other rows, and the host half of B200FlatIndex's "filter": "exact" mode (filter_ids -> rows, k not 2k,
min(k, |allowed|) ids) with the device index swapped for an oracle-backed stand-in."""
import numpy as np
import pytest

from oracle.flat_ip import FLT_MAX, IndexFlatIP, normalize_L2


def oracle_allowed(xb, q, k, mask):
    """Exact top-k over the rows where `mask` (bool, length <= len(xb)) is True: the oracle searches those rows alone and
    the ids are mapped back; the row list is ascending, so the (score desc, row asc) order is kept.  -1 / -FLT_MAX pad."""
    rows = np.flatnonzero(mask)
    D = np.full((len(q), k), -FLT_MAX, np.float32)
    I = np.full((len(q), k), -1, np.int64)
    if rows.size:
        ix = IndexFlatIP(xb.shape[1])
        ix.add(xb[rows])
        D, i = ix.search(q, k)
        I = np.where(i >= 0, rows[np.maximum(i, 0)], -1)
    return D, I


def _brute(xb, q, k, allow):
    s = q.astype(np.float64) @ xb.astype(np.float64).T
    D = np.full((len(q), k), -FLT_MAX, np.float32)
    I = np.full((len(q), k), -1, np.int64)
    rows = np.flatnonzero(allow)
    for r in range(len(q)):
        order = rows[np.lexsort((rows, -s[r, rows]))][:k]
        D[r, :len(order)] = s[r, order]
        I[r, :len(order)] = order
    return D, I


@pytest.mark.parametrize("n_allowed", [0, 1, 9, 250, 1000])
def test_filtered_oracle_equals_brute_force_on_massive_ties(n_allowed):
    """Integer data (exact fp32 scores) with a handful of distinct values: the order inside ties is row ascending, the
    padding past the allowed rows is -1 / -FLT_MAX, disallowed rows never appear, and the result equals the oracle's own
    exclusion masking (scripts/evaluate_model.py's -inf mask) applied to every disallowed row."""
    rng = np.random.default_rng(n_allowed)
    N, d, k = 1000, 8, 10
    xb = rng.integers(-1, 2, size=(N, d)).astype(np.float32)
    q = rng.integers(-1, 2, size=(7, d)).astype(np.float32)
    allow = np.zeros(N, bool)
    allow[rng.permutation(N)[:n_allowed]] = True
    ix = IndexFlatIP(d, db_block=300)
    ix.add(xb)
    D, I = oracle_allowed(xb, q, k, allow)
    bD, bI = _brute(xb, q, k, allow)
    assert np.array_equal(I, bI) and np.array_equal(D, bD)
    eD, eI = ix.search(q, k, exclude=[np.flatnonzero(~allow)] * len(q))
    assert np.array_equal(I, eI) and np.array_equal(D, eD)
    assert (I[:, min(k, n_allowed):] == -1).all() and (D[:, min(k, n_allowed):] == -FLT_MAX).all()
    if n_allowed == N:
        uD, uI = ix.search(q, k)
        assert np.array_equal(D, uD) and np.array_equal(I, uI)
        assert D.tobytes() == uD.tobytes()
    # a mask shorter than the catalogue leaves the missing tail out
    D2, I2 = oracle_allowed(xb, q, k, allow[:600])
    bD2, bI2 = _brute(xb, q, k, np.concatenate([allow[:600], np.zeros(400, bool)]))
    assert np.array_equal(I2, bI2) and np.array_equal(D2, bD2)


class _OracleFilter:
    def __init__(self, mask):
        self.mask = mask


class _OracleDeviceIndex:
    """CPU stand-in for b200rec.retrieval.FlatIPDeviceIndex in HOST-LOGIC tests only: `add`, `search(q, k, normalize,
    sel)`, `row_filter(rows=)`, `ntotal`, `reconstruct_n`, a filtered search answered by `oracle_allowed`."""

    def __init__(self, d, storage="fp32", device=None, row_offset=0):
        self.d, self._ix = d, IndexFlatIP(d)

    ntotal = property(lambda self: self._ix.ntotal)

    def add(self, x, normalize=False):
        x = np.array(x, dtype=np.float32)
        self._ix.add(normalize_L2(x) if normalize else x)

    def row_filter(self, rows=None, mask=None):
        r = np.asarray(rows, dtype=np.int64).reshape(-1)
        m = np.zeros(self.ntotal, bool)
        m[r[(r >= 0) & (r < self.ntotal)]] = True
        return _OracleFilter(m)

    def search(self, q, k, normalize=False, sel=None):
        q = np.array(q, dtype=np.float32).reshape(-1, self.d)
        q = normalize_L2(q) if normalize else q
        return self._ix.search(q, k) if sel is None else oracle_allowed(self._ix.xb, q, k, sel.mask)

    def reconstruct_n(self, i0=0, n=None):
        return self._ix.xb[i0:(None if n is None else i0 + n)].copy()


@pytest.mark.parametrize("metric", ["cosine", "ip"])
def test_exact_filter_mode_host_logic(monkeypatch, metric):
    from b200rec import retrieval
    monkeypatch.setattr(retrieval, "FlatIPDeviceIndex", _OracleDeviceIndex)
    rng = np.random.default_rng(5)
    N, D, k = 300, 16, 10
    emb = rng.standard_normal((N, D)).astype(np.float32)
    qry = rng.standard_normal((4, D)).astype(np.float32)
    names = [f"item_{i}" for i in range(N)]
    with pytest.raises(ValueError, match="filter"):
        retrieval.B200FlatIndex({"dimension": D, "filter": "pre"})
    post = retrieval.B200FlatIndex({"dimension": D, "metric": metric})
    exact = retrieval.B200FlatIndex({"dimension": D, "metric": metric, "filter": "exact"})
    post.build(emb.copy(), names)
    exact.build(emb.copy(), names)

    def want(allowed_rows, kk):
        mask = np.zeros(N, bool)
        mask[list(allowed_rows)] = True
        q = normalize_L2(qry.copy()) if metric == "cosine" else qry
        Dr, Ir = oracle_allowed(normalize_L2(emb.copy()) if metric == "cosine" else emb, q, kk, mask)
        return ([[names[i] for i in row if i >= 0] for row in Ir],
                [[float(s) for s, i in zip(ds, row) if i >= 0] for ds, row in zip(Dr, Ir)])

    allowed = rng.permutation(N)[:40]
    fids = [names[i] for i in allowed] + ["unknown_1", names[allowed[0]], names[allowed[3]], "zzz"]   # unknown + duplicates
    ids, scores = exact.search(qry.copy(), k=k, filter_ids=fids)
    w_ids, w_scores = want(allowed, k)
    assert ids == w_ids and all(len(r) == k for r in ids)
    for a, b in zip(scores, w_scores):
        assert np.allclose(a, b, rtol=0, atol=0)
    assert all(set(r) <= set(fids) for r in ids)
    # fewer allowed rows than k: min(k, |allowed|) ids, in oracle order
    few = [names[7], names[123], names[299], "nope"]
    ids, _ = exact.search(qry.copy(), k=k, filter_ids=few)
    assert ids == want([7, 123, 299], k)[0] and all(len(r) == 3 for r in ids)
    # a selective filter: the post-pass over the 2k best rows loses results, the exact mode does not
    sel = [names[i] for i in allowed[:20]]
    p_ids, _ = post.search(qry.copy(), k=k, filter_ids=sel)
    e_ids, _ = exact.search(qry.copy(), k=k, filter_ids=sel)
    assert all(len(r) == k for r in e_ids) and sum(map(len, p_ids)) < sum(map(len, e_ids))
    # [] allows nothing in both modes; no filter is the plain search in both modes
    assert exact.search(qry[:2].copy(), k=4, filter_ids=[]) == ([[], []], [[], []])
    assert post.search(qry[:2].copy(), k=4, filter_ids=[]) == ([[], []], [[], []])
    assert exact.search(qry.copy(), k=k) == post.search(qry.copy(), k=k)
    # rows added later are reachable through their ids
    exact.add(rng.standard_normal((5, D)).astype(np.float32), [f"new_{i}" for i in range(5)])
    ids, _ = exact.search(qry.copy(), k=3, filter_ids=["new_2", "new_4"])
    assert all(sorted(r) == ["new_2", "new_4"] for r in ids)
