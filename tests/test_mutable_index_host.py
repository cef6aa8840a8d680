"""CPU checks of the mutable catalogue (no GPU): the host bookkeeping of B200FlatIndex under "updates": "in_place"
(upsert / remove / slot reuse / id maps / save -> load / compact / both filter_ids modes / RetrievalEngine) with the
device index swapped for an oracle-backed stand-in that implements update_rows / remove_rows / compact, the "warn"
default (the reference's warnings, nothing changes), and FlatIPDeviceIndex's host validation of mutation arguments,
which must raise before any device work."""
import heapq
import logging

import numpy as np
import pytest
import torch

from oracle.flat_ip import FLT_MAX, IndexFlatIP, normalize_L2


class _OracleMutableIndex:
    """CPU stand-in for FlatIPDeviceIndex in HOST-LOGIC tests only: row slots (xb) + live mask, searched with the oracle
    over the live (and filter-allowed) rows alone, ids mapped back through the ascending row list."""

    def __init__(self, d, storage="fp32", device=None, row_offset=0):
        self.d = d
        self.xb = np.zeros((0, d), np.float32)
        self.live = np.zeros(0, bool)
        self.calls = []

    ntotal = property(lambda self: len(self.xb))
    n_live = property(lambda self: int(self.live.sum()))

    def add(self, x, normalize=False):
        x = np.array(x, dtype=np.float32)
        self.calls.append(("add", len(x)))
        self.xb = np.concatenate([self.xb, normalize_L2(x) if normalize else x])
        self.live = np.concatenate([self.live, np.ones(len(x), bool)])

    def update_rows(self, rows, x, normalize=False):
        rows = np.asarray(rows)
        assert rows.dtype == np.int64 and len(set(rows.tolist())) == len(rows) and ((rows >= 0) & (rows < self.ntotal)).all()
        x = np.array(x, dtype=np.float32)
        self.calls.append(("update_rows", len(rows)))
        self.xb[rows] = normalize_L2(x) if normalize else x
        self.live[rows] = True

    def remove_rows(self, rows):
        rows = np.unique(np.asarray(rows))
        self.calls.append(("remove_rows", len(rows)))
        n = int(self.live[rows].sum())
        self.live[rows] = False
        return n

    def compact(self):
        keep = np.flatnonzero(self.live)
        remap = np.full(self.ntotal, -1, np.int64)
        remap[keep] = np.arange(keep.size)
        self.xb, self.live = self.xb[keep], np.ones(keep.size, bool)
        return remap

    def row_filter(self, rows=None, mask=None):
        return np.unique(np.asarray(rows, dtype=np.int64))

    def search(self, q, k, normalize=False, sel=None):
        q = np.array(q, dtype=np.float32).reshape(-1, self.d)
        q = normalize_L2(q) if normalize else q
        mask = self.live.copy()
        if sel is not None:
            allowed = np.zeros(self.ntotal, bool)
            allowed[sel] = True
            mask &= allowed
        rows = np.flatnonzero(mask)
        D = np.full((len(q), k), -FLT_MAX, np.float32)
        I = np.full((len(q), k), -1, np.int64)
        if rows.size:
            ix = IndexFlatIP(self.d)
            ix.add(self.xb[rows])
            D, i = ix.search(q, k)
            I = np.where(i >= 0, rows[np.maximum(i, 0)], -1)
        return D, I

    def reconstruct_n(self, i0=0, n=None):
        return self.xb[i0:(None if n is None else i0 + n)].copy()


@pytest.fixture
def stand_in(monkeypatch):
    from b200rec import retrieval
    monkeypatch.setattr(retrieval, "FlatIPDeviceIndex", _OracleMutableIndex)
    return retrieval


def _check_maps(ix):
    assert len(ix.id_map) == len(ix.reverse_id_map) == ix.current_size == ix.index.n_live
    for row, item_id in ix.id_map.items():
        assert ix.reverse_id_map[item_id] == row and 0 <= row < ix.index.ntotal and ix.index.live[row]
    assert sorted(ix._free) == sorted(set(range(ix.index.ntotal)) - set(ix.id_map))
    assert ix._free == sorted(ix._free) or ix._free[0] == min(ix._free)        # a heap: lowest free slot first


def _same_as_fresh(retrieval, ix, live, qry, k, metric):
    fresh = retrieval.B200FlatIndex({"dimension": qry.shape[1], "metric": metric})
    names = sorted(live)
    fresh.build(np.stack([live[n] for n in names]), names)
    got, want = ix.search(qry, k=k), fresh.search(qry, k=k)
    assert got[0] == want[0]
    for a, b in zip(got[1], want[1]):
        assert np.allclose(a, b, rtol=1e-6, atol=1e-6)


@pytest.mark.parametrize("metric", ["cosine", "ip"])
def test_random_upsert_remove_readd_sequences_keep_the_maps_and_equal_a_fresh_index(stand_in, metric):
    retrieval = stand_in
    rng = np.random.default_rng(3 if metric == "ip" else 4)
    D, k = 16, 12
    ix = retrieval.B200FlatIndex({"dimension": D, "metric": metric, "updates": "in_place"})
    live = {f"i{j}": rng.standard_normal(D).astype(np.float32) for j in range(200)}
    names = list(live)
    ix.build(np.stack([live[n] for n in names]), names)
    qry = rng.standard_normal((5, D)).astype(np.float32)
    universe = [f"i{j}" for j in range(320)]
    for step in range(40):
        op = rng.integers(0, 3)
        if op == 0:                                        # upsert with repeats inside one call: last occurrence wins
            ids = [universe[j] for j in rng.integers(0, len(universe), size=int(rng.integers(1, 25)))]
            emb = rng.standard_normal((len(ids), D)).astype(np.float32)
            before_free, before_n = len(ix._free), ix.index.ntotal
            n_new = len({x for x in ids if x not in ix.reverse_id_map})
            (ix.add if step % 2 else ix.update)(emb, ids)
            for x, e in zip(ids, emb):
                live[x] = e
            assert ix.index.ntotal == before_n + max(0, n_new - before_free)      # removed slots are reused first
        else:
            ids = [universe[j] for j in rng.integers(0, len(universe), size=int(rng.integers(1, 30)))]
            known = {x for x in ids if x in ix.reverse_id_map}
            rows = sorted(ix.reverse_id_map[x] for x in known)
            assert ix.remove(ids + ids[:3]) == len(known)
            for x in known:
                del live[x]
            assert all(ix.index.live[r] == False for r in rows)                   # noqa: E712
        _check_maps(ix)
        assert set(ix.reverse_id_map) == set(live)
        if step % 5 == 4:
            _same_as_fresh(retrieval, ix, live, qry, k, metric)
    _same_as_fresh(retrieval, ix, live, qry, min(k, len(live)), metric)
    res = ix.search(qry, k=k)[0]
    assert all(len(set(r)) == len(r) for r in res)                                # no item twice in a result list


def test_new_ids_fill_removed_slots_lowest_first_then_append(stand_in):
    ix = stand_in.B200FlatIndex({"dimension": 4, "metric": "ip", "updates": "in_place"})
    ix.build(np.eye(4, dtype=np.float32)[[0, 1, 2, 3, 0, 1]] * np.arange(1, 7)[:, None], list("abcdef"))
    assert ix.remove(["e", "b", "zz", "b"]) == 2
    assert ix.current_size == 4 and ix._free == [1, 4]
    ix.add(np.ones((3, 4), np.float32), ["x", "y", "z"])
    assert (ix.reverse_id_map["x"], ix.reverse_id_map["y"], ix.reverse_id_map["z"]) == (1, 4, 6)
    assert ix.index.ntotal == 7 and ix.current_size == 7
    ix.update(np.full((2, 4), 2.0, np.float32), ["x", "x"])                      # a known id: in place, no new slot
    assert ix.index.ntotal == 7 and ix.reverse_id_map["x"] == 1 and np.all(ix.index.xb[1] == 2.0)
    with pytest.raises(ValueError):
        ix.add(np.ones((2, 4), np.float32), ["only_one"])


def test_build_with_a_repeated_id_keeps_its_last_row(stand_in):
    ix = stand_in.B200FlatIndex({"dimension": 2, "metric": "ip", "updates": "in_place"})
    ix.build(np.array([[1, 0], [2, 0], [3, 0]], np.float32), ["a", "b", "a"])
    assert ix.reverse_id_map == {"a": 2, "b": 1} and ix.current_size == 2 and ix._free == [0]
    assert ix.search(np.array([1, 0], np.float32), k=3)[0] == [["a", "b"]]


@pytest.mark.parametrize("mode", ["post", "exact"])
def test_filter_modes_work_over_live_rows(stand_in, mode):
    rng = np.random.default_rng(11)
    D, N = 8, 60
    ix = stand_in.B200FlatIndex({"dimension": D, "metric": "ip", "updates": "in_place", "filter": mode})
    emb = rng.standard_normal((N, D)).astype(np.float32)
    names = [f"n{j}" for j in range(N)]
    ix.build(emb, names)
    ix.remove(names[::3])
    q = rng.standard_normal((4, D)).astype(np.float32)
    fids = names[:40]
    ids, _ = ix.search(q, k=5, filter_ids=fids)
    gone = set(names[::3])
    assert all(set(r) <= set(fids) - gone for r in ids)
    if mode == "exact":
        assert all(len(r) == 5 for r in ids)


def test_save_load_writes_the_live_rows_densely(stand_in, tmp_path):
    from b200rec.retrieval import read_ixfi
    rng = np.random.default_rng(5)
    D = 8
    ix = stand_in.B200FlatIndex({"dimension": D, "metric": "cosine", "updates": "in_place"})
    names = [f"n{j}" for j in range(30)]
    ix.build(rng.standard_normal((30, D)).astype(np.float32), names)
    ix.remove(names[5:12])
    ix.add(rng.standard_normal((3, D)).astype(np.float32), ["n1", "new0", "new1"])
    q = rng.standard_normal((3, D)).astype(np.float32)
    want = ix.search(q, k=10)
    ix.save(str(tmp_path / "m"))
    rows = read_ixfi(tmp_path / "m.faiss")
    assert rows.shape == (ix.current_size, D)
    ix2 = stand_in.B200FlatIndex({"dimension": D, "metric": "cosine", "updates": "in_place"})
    ix2.load(str(tmp_path / "m"))
    assert ix2.current_size == ix.current_size and ix2.index.ntotal == ix.current_size and ix2._free == []
    assert sorted(ix2.id_map) == list(range(ix.current_size)) and set(ix2.reverse_id_map) == set(ix.reverse_id_map)
    for item_id, row in ix2.reverse_id_map.items():
        assert np.array_equal(rows[row], ix.index.xb[ix.reverse_id_map[item_id]])
    got = ix2.search(q, k=10)
    assert got[0] == want[0] and np.allclose(got[1], want[1])


def test_compact_renumbers_the_id_maps(stand_in):
    rng = np.random.default_rng(6)
    ix = stand_in.B200FlatIndex({"dimension": 4, "metric": "ip", "updates": "in_place"})
    names = [f"n{j}" for j in range(20)]
    ix.build(rng.standard_normal((20, 4)).astype(np.float32), names)
    ix.remove(names[::4])
    q = rng.standard_normal((3, 4)).astype(np.float32)
    want = ix.search(q, k=8)
    remap = ix.compact()
    assert (remap[::4] == -1).all() and ix.index.ntotal == 15 and ix._free == []
    assert sorted(ix.id_map) == list(range(15)) and ix.current_size == 15
    assert ix.search(q, k=8) == want
    _check_maps(ix)


def test_engine_stream_of_updates_and_removals(stand_in):
    rng = np.random.default_rng(8)
    D = 8
    eng = stand_in.RetrievalEngine({"index_type": "b200", "embedding_dim": D, "b200": {"metric": "cosine",
                                                                                        "updates": "in_place"}})
    names = [f"n{j}" for j in range(50)]
    eng.build_index(rng.standard_normal((50, D)).astype(np.float32), names)
    q = rng.standard_normal((4, D)).astype(np.float32)
    sizes = []
    for step in range(30):                                  # Kafka-like: re-embedded items, a few removals, new items
        ids = [names[j] for j in rng.integers(0, 50, size=6)] + [f"new{step}"]
        eng.update_index(rng.standard_normal((len(ids), D)).astype(np.float32), ids)
        eng.index.remove([f"new{step - 1}", names[int(rng.integers(0, 50))]])
        out, _, _ = eng.retrieve(q, k=20)
        assert all(len(set(r)) == len(r) for r in out)
        assert eng.get_metrics()["index_size"] == eng.index.current_size == eng.index.index.n_live
        sizes.append(eng.index.index.ntotal)
    assert sizes[-1] == sizes[10]                           # slots are reused: the catalogue stops growing


def test_warn_default_logs_and_changes_nothing(stand_in, caplog):
    ix = stand_in.B200FlatIndex({"dimension": 4, "metric": "ip"})
    assert ix.updates == "warn"
    ix.build(np.eye(4, dtype=np.float32), list("abcd"))
    calls = list(ix.index.calls)
    with caplog.at_level(logging.WARNING, logger="b200rec"):
        assert ix.update(np.ones((1, 4), np.float32), ["a"]) is None
        assert ix.remove(["a"]) is None
    assert "do not support in-place updates" in caplog.text and "do not support removal" in caplog.text
    assert ix.index.calls == calls and ix.current_size == 4 and ix.reverse_id_map["a"] == 0
    ix.add(np.ones((1, 4), np.float32), ["a"])              # the reference appends a second row for a known id
    assert ix.index.ntotal == 5 and ix.current_size == 5 and ix.reverse_id_map["a"] == 4 and ix.id_map[0] == "a"
    with pytest.raises(ValueError, match="updates"):
        stand_in.B200FlatIndex({"dimension": 4, "updates": "sometimes"})


def test_device_index_validates_mutation_arguments_before_any_device_work(monkeypatch):
    """FlatIPDeviceIndex.update_rows / remove_rows check rows and shapes on the host: the object is built without a GPU
    and every kernel wrapper is replaced by one that fails, so a call that got past validation would raise differently."""
    from b200rec import kernels as K
    from b200rec.retrieval import FlatIPDeviceIndex

    def boom(*a, **kw):
        raise AssertionError("device work before validation")
    for name in ("update_rows", "clear_row_bits", "patch_compacted", "rows_to_bitmap"):
        monkeypatch.setattr(K, name, boom)
    ix = FlatIPDeviceIndex.__new__(FlatIPDeviceIndex)
    ix.ntotal, ix.d = 10, 4
    x = np.zeros((2, 4), np.float32)
    for bad in ([3, 10], [-1, 2], np.array([1.0, 2.0]), np.array([[1, 2]]), torch.tensor([0, 11])):
        with pytest.raises(ValueError):
            ix.update_rows(bad, x)
        with pytest.raises(ValueError):
            ix.remove_rows(bad)
    for shape in ((3, 4), (2, 5), (8,)):
        with pytest.raises(ValueError):
            ix.update_rows([1, 2], np.zeros(shape, np.float32))
    ix.update_rows([], np.zeros((0, 4), np.float32))        # empty calls are no-ops
    assert ix.remove_rows(np.zeros(0, np.int64)) == 0
