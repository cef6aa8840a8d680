"""Every kernel instantiation and work decomposition of exact top-K search against the oracle, bit for bit.

Each case first proves, through the plan query, that its shape and development knobs reach the instantiation named in
its id (a shape that silently falls back to another path fails), then compares scores and ids with
`oracle.flat_ip.IndexFlatIP` under the total order (score desc, row asc).  The data are integers in [-3, 3]: exact in
bf16, with exact fp32 scores (|s| <= 9 * 704), so ties are everywhere and only the exact order passes.

Instantiations (tests/topk_plan.py names them): pair2 / pair1 = the 2-CTA pair kernel with 512 / 256 queries per
supertile (-ks1: one 64-column atom per ring stage, odd ld / 64), nq2bn128 = single-CTA kernel with 256 resident
queries and 128-row tiles, bn256 / bn64 = single-CTA kernel with 128 resident queries and 256- / 64-row tiles."""
import functools
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from topk_plan import DEFAULT_MAP, KNOBS, default_path, path_name, plan, topk_knobs  # noqa: E402

pytestmark = pytest.mark.gpu

FLT_MAX = float(np.finfo(np.float32).max)
N_MAP = 50_000 + 37

# one reachable shape per instantiation: (ld, Q, knobs)
PATHS = {
    "pair2": (128, 300, {}),
    "pair1": (128, 200, {}),
    "pair1-ks1": (448, 200, {}),
    "nq2bn128": (64, 200, {"B200REC_TOPK_V2": 0}),
    "bn256": (64, 100, {}),
    "bn64": (512, 100, {}),
}
TILE_ROWS = {"pair2": 128, "pair1": 256, "pair1-ks1": 256, "nq2bn128": 128, "bn256": 256, "bn64": 64}
# knobs that put a path's kernel on Q = 200 / Q = 600 (both sides of the k > 128 && Q <= 256 flush rule)
AT_Q = {
    "pair2": {200: {"B200REC_TOPK_V2": 2}, 600: {}},
    "pair1-ks1": {200: {}, 600: {}},
    "bn256": {200: {"B200REC_TOPK_V2": 0, "B200REC_TOPK_NQ": 1}, 600: {"B200REC_TOPK_V2": 0, "B200REC_TOPK_NQ": 1}},
    "bn64": {200: {}, 600: {}},
}


@pytest.fixture
def knobs():
    """topk_knobs(**env): development knobs for a block, restored (environment and library) on exit."""
    saved = {name: os.environ.get(name) for name in KNOBS}
    yield topk_knobs
    assert {name: os.environ.get(name) for name in KNOBS} == saved


@pytest.fixture(autouse=True, scope="module")
def _default_plans():
    if plan(N_MAP, 64, 1, 10)["sms"] != 148:
        pytest.skip("the instantiation map is pinned for 148 SMs")
    yield
    _cat_dev.cache_clear()


@functools.lru_cache(maxsize=8)
def _cat(n: int, ld: int) -> np.ndarray:
    return np.random.default_rng([n, ld]).integers(-3, 4, size=(n, ld), dtype=np.int8).astype(np.float32)


@functools.lru_cache(maxsize=4)
def _cat_dev(n: int, ld: int) -> torch.Tensor:
    return torch.from_numpy(_cat(n, ld)).cuda().to(torch.bfloat16)


def _qry(q: int, ld: int) -> np.ndarray:
    """The first q rows of a fixed pool, so results for fewer queries are row slices of one oracle call."""
    return np.random.default_rng([ld, 7]).integers(-3, 4, size=(1024, ld), dtype=np.int8)[:q].astype(np.float32)


def _qry_dev(q: int, ld: int) -> torch.Tensor:
    return torch.from_numpy(_qry(q, ld)).cuda().to(torch.bfloat16)


def _oracle(cat: np.ndarray, qry: np.ndarray, k: int, exclude=None):
    from oracle.flat_ip import IndexFlatIP
    ix = IndexFlatIP(cat.shape[1])
    ix.add(cat)
    return ix.search(qry, k, exclude=exclude)


@functools.lru_cache(maxsize=16)
def _ref(n: int, ld: int, q: int, k: int):
    return _oracle(_cat(n, ld), _qry(q, ld), k)


def _assert_exact(D, I, rD, rI, what: str) -> None:
    D = D.cpu().numpy() if torch.is_tensor(D) else D
    I = I.cpu().numpy() if torch.is_tensor(I) else I
    assert D.shape == rD.shape and I.shape == rI.shape, what
    bad = np.argwhere((D != rD) | (I != rI))
    if bad.size:
        qi, j = bad[0]
        raise AssertionError(f"{what}: {len(bad)} of {D.size} slots differ; first: query {qi} rank {j} got "
                             f"({D[qi, j]}, {I[qi, j]}) want ({rD[qi, j]}, {rI[qi, j]})")


def _expect_path(name: str, n: int, ld: int, q: int, k: int, shards: int = 1) -> dict:
    p = plan(n, ld, q, k, shards)
    assert path_name(p) == name, f"(N={n}, ld={ld}, Q={q}, k={k}) plans {path_name(p)}, not {name}: {p}"
    return p


def _search(name, n, ld, q, k, **kw):
    from b200rec import kernels as KR
    p = _expect_path(name, n, ld, q, k)
    D, I = KR.flat_ip_topk(_cat_dev(n, ld), _qry_dev(q, ld), k, **kw)
    torch.cuda.synchronize()
    return p, D, I


# ------------------------------------------------------------------------------------------------ default map
MAP_CASES = [(ld, q) for ld in sorted(DEFAULT_MAP) if ld in (64, 128, 256, 320, 384, 448, 512, 576, 704)
             for q in (1, 128, 129, 256, 257, 513)]


@pytest.mark.parametrize("ld,q", MAP_CASES, ids=[f"{default_path(ld, q)}-ld{ld}-q{q}" for ld, q in MAP_CASES])
def test_default_map(ld, q):
    rD, rI = _ref(N_MAP, ld, 513, 10)
    _, D, I = _search(default_path(ld, q), N_MAP, ld, q, 10)
    _assert_exact(D, I, rD[:q], rI[:q], f"ld={ld} Q={q}")


# ------------------------------------------------------------------------------------------------ forced paths
FORCED = [("nq2bn128", 64, 129, {"B200REC_TOPK_V2": 0}), ("nq2bn128", 64, 600, {"B200REC_TOPK_V2": 0}),
          ("nq2bn128", 256, 129, {"B200REC_TOPK_V2": 0}), ("nq2bn128", 256, 600, {"B200REC_TOPK_V2": 0}),
          ("pair2", 128, 200, {"B200REC_TOPK_V2": 2}), ("pair1", 128, 600, {"B200REC_TOPK_V2": 1}),
          ("bn256", 64, 600, {"B200REC_TOPK_V2": 0, "B200REC_TOPK_NQ": 1})]


@pytest.mark.parametrize("name,ld,q,env", FORCED, ids=[f"{c[0]}-ld{c[1]}-q{c[2]}" for c in FORCED])
def test_forced_instantiation(knobs, name, ld, q, env):
    assert default_path(ld, q) != name
    rD, rI = _ref(N_MAP, ld, q, 10)
    with knobs(**env):
        _, D, I = _search(name, N_MAP, ld, q, 10)
    _assert_exact(D, I, rD, rI, f"{name} ld={ld} Q={q}")


# ------------------------------------------------------------------------------------------------ k edges
K_PATHS = ("pair2", "pair1-ks1", "bn256", "bn64")
K_EDGES = (1, 2, 32, 33, 255, 256, 257, 1024, 1025, 2048)


@pytest.mark.parametrize("k", K_EDGES)
@pytest.mark.parametrize("name", K_PATHS)
def test_k_edges(name, k):
    ld, q, env = PATHS[name]
    assert not env
    n = 20_000
    rD, rI = _ref(n, ld, q, k)
    _, D, I = _search(name, n, ld, q, k)
    _assert_exact(D, I, rD, rI, f"{name} k={k}")


@pytest.mark.parametrize("q", (200, 600))
@pytest.mark.parametrize("name", K_PATHS)
def test_k_1025_both_sides_of_the_flush_rule(knobs, name, q):
    ld = PATHS[name][0]
    n, k = 20_000, 1025
    rD, rI = _ref(n, ld, q, k)
    with knobs(**AT_Q[name][q]):
        p, D, I = _search(name, n, ld, q, k)
    assert p["flush"] == (p["cap"] if q <= 256 else 256), p
    _assert_exact(D, I, rD, rI, f"{name} Q={q} k={k}")


@pytest.mark.parametrize("name", K_PATHS)
def test_k_larger_than_catalogue_pads(name):
    ld, q, _ = PATHS[name]
    n, k = 1500, 2048
    rD, rI = _ref(n, ld, q, k)
    _, D, I = _search(name, n, ld, q, k)
    D, I = D.cpu().numpy(), I.cpu().numpy()
    assert (I[:, n:] == -1).all() and (D[:, n:] == -FLT_MAX).all()
    assert (np.sort(I[:, :n], axis=1) == np.arange(n)).all()
    _assert_exact(D, I, rD, rI, f"{name} N={n} k={k}")


# ------------------------------------------------------------------------------------------------ N edges
def _n_edges(name):
    bn = TILE_ROWS[name]
    return [1, bn - 1, bn, bn + 1, 2 * bn + 1]


N_CASES = [(name, n) for name in PATHS for n in _n_edges(name)] + [("pair2", 9_000), ("pair1", 18_000)]


@pytest.mark.parametrize("name,n", N_CASES, ids=[f"{c[0]}-N{c[1]}" for c in N_CASES])
def test_n_edges(knobs, name, n):
    ld, q, env = PATHS[name]
    k = 10
    rD, rI = _ref(n, ld, q, k)
    with knobs(**env):
        p, D, I = _search(name, n, ld, q, k)
    if n > 2 * TILE_ROWS[name] + 1:      # the pair kernel with fewer tiles than CTA pairs: one unit per tile
        assert p["S"] * p["T"] < p["sms"] // 2 and p["grid"] == 2 * p["S"] * p["T"], p
    _assert_exact(D, I, rD, rI, f"{name} N={n}")


# ------------------------------------------------------------------------------------------------ threshold start
@pytest.mark.parametrize("start", ("sample", "nosample", "tau-two-shards", "row-offset"))
@pytest.mark.parametrize("name", list(PATHS))
def test_threshold_start(knobs, name, start):
    from b200rec import kernels as KR
    ld, q, env = PATHS[name]
    n, k = N_MAP, 10
    rD, rI = _ref(n, ld, q, k)
    if start == "nosample":
        env = {**env, "B200REC_TOPK_NOSAMPLE": 1}
    with knobs(**env):
        if start in ("sample", "nosample"):
            p, D, I = _search(name, n, ld, q, k)
            assert (p["sample_m"] > 0) == (start == "sample"), p
            _assert_exact(D, I, rD, rI, f"{name} {start}")
        elif start == "row-offset":
            off = 1 << 33
            _, D, I = _search(name, n, ld, q, k, row_offset=off)
            _assert_exact(D, I, rD, rI + off, f"{name} row_offset")
        else:
            cat, qd = _cat_dev(n, ld), _qry_dev(q, ld)
            halves = ((0, 20_011), (20_011, n))
            vals = []
            for lo, hi in halves:
                p = _expect_path(name, hi - lo, ld, q, k, shards=2)
                assert p["sample_m"] > 0, p
                ws = torch.empty((KR.topk_workspace_bytes(hi - lo, ld, q, k),), dtype=torch.uint8, device="cuda")
                vals.append(KR.topk_sample(cat[lo:hi], qd, k, ws, k, 2))
            tau = KR.topk_pooled_kth(torch.stack(vals).contiguous(), k)
            assert (tau.cpu().numpy() <= rD[:, k - 1]).all(), "pooled threshold above the k-th score"
            parts = [KR.flat_ip_topk(cat[lo:hi], qd, k, row_offset=lo, tau_init=tau) for lo, hi in halves]
            D, I = KR.topk_merge(torch.stack([d for d, _ in parts]).contiguous(),
                                 torch.stack([i for _, i in parts]).contiguous(), k)
            torch.cuda.synchronize()
            _assert_exact(D, I, rD, rI, f"{name} tau_init over two shards")


# ------------------------------------------------------------------------------------------------ allow-lists, exclusion
@pytest.mark.parametrize("mode", ("bitmap-0.9", "bitmap-0.05", "compact-0.05", "exclude"))
@pytest.mark.parametrize("name", ("pair1-ks1", "bn64"))
def test_allow_lists_and_exclusion(name, mode):
    from b200rec import kernels as KR
    ld, q, _ = PATHS[name]
    n, k = N_MAP, 10
    cat, qry = _cat(n, ld), _qry(q, ld)
    rng = np.random.default_rng([n, ld, q])
    if mode == "exclude":
        top = _ref(n, ld, q, k)[1]
        excl = [np.unique(np.concatenate([top[i, : i % 5], rng.choice(n, size=rng.integers(0, 300), replace=False)]))
                .astype(np.int32) for i in range(q)]
        rD, rI = _oracle(cat, qry, k, exclude=excl)
        indptr = torch.tensor(np.concatenate([[0], np.cumsum([len(e) for e in excl])]), dtype=torch.int64, device="cuda")
        _, D, I = _search(name, n, ld, q, k, exclude_indptr=indptr,
                          exclude_rows=torch.from_numpy(np.concatenate(excl)).cuda())
        _assert_exact(D, I, rD, rI, f"{name} exclusion lists")
        return
    frac = float(mode.split("-")[1])
    rows = np.flatnonzero(rng.random(n) < frac)
    rD, rI = _oracle(cat[rows], qry, k)
    rI = np.where(rI >= 0, rows[np.maximum(rI, 0)], -1)
    rows_d = torch.from_numpy(rows).cuda()
    if mode.startswith("bitmap"):
        _expect_path(name, n, ld, q, k)
        D, I = KR.flat_ip_topk_filtered(_cat_dev(n, ld), _qry_dev(q, ld), k, KR.rows_to_bitmap(rows_d, n), n)
    else:
        _expect_path(name, rows.size, ld, q, k)
        D, I = KR.flat_ip_topk(_cat_dev(n, ld)[rows_d].contiguous(), _qry_dev(q, ld), k)
        KR.remap_ids(I, rows_d)
    torch.cuda.synchronize()
    _assert_exact(D, I, rD, rI, f"{name} {mode}")


# ------------------------------------------------------------------------------------------------ through the index
@pytest.mark.parametrize("q", (100, 300))
@pytest.mark.parametrize("d", (160, 192))
def test_fp32_storage_index(d, q):
    """fp32 storage searches 3 bf16 pieces per value: ld = 576, the BN = 64 kernel at Q <= 128 and the pair kernel with
    one atom per stage above, selecting k + margin candidates that are re-scored from the fp32 rows."""
    from b200rec.retrieval import FlatIPDeviceIndex
    n, k = 30_000, 10
    ix = FlatIPDeviceIndex(d, storage="fp32")
    assert ix.ld == 576
    cat = _cat(n, 192)[:, :d].copy()
    qry = _qry(q, 192)[:, :d].copy()
    ix.add(cat)
    k_in = min(k + ix.rescore_margin(k), max(k, min(n, 2048)))
    _expect_path("bn64" if q <= 128 else "pair1-ks1", n, 576, q, k_in)
    D, I = ix.search(qry, k)
    rD, rI = _oracle(cat, qry, k)
    _assert_exact(D, I, rD, rI, f"fp32 storage d={d} Q={q}")


def test_bf16_storage_index_beyond_the_fp32_limit():
    from b200rec.retrieval import FlatIPDeviceIndex
    n, q, k, d = 30_000, 100, 10, 256
    with pytest.raises(ValueError, match="storage='bf16'"):
        FlatIPDeviceIndex(d)
    ix = FlatIPDeviceIndex(d, storage="bf16")
    ix.add(_cat(n, d))
    _expect_path("bn256", n, d, q, k)
    D, I = ix.search(_qry(q, d), k)
    rD, rI = _ref(n, d, q, k)
    _assert_exact(D, I, rD, rI, "bf16 storage d=256")
