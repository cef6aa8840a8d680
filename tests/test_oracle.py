"""CPU tests: pin the oracle (oracle/) against the golden vectors produced by the imported reference
(tests/golden/make_golden.py) and against the reference's own exact-retrieval twin."""
import glob
import os

import numpy as np
import pytest

from oracle import flat_ip, two_tower as tt


def _tower(g, prefix, L, act="relu"):
    params = {k[len(prefix) + 1:]: g[k] for k in g.files if k.startswith(prefix + ".")}
    return tt.TowerOracle(params, L, act)


@pytest.mark.parametrize("name", ["step_ml1m", "step_small"])
def test_trainer_step_matches_reference(golden_dir, name):
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    T = float(g["temperature"])
    ut, it = _tower(g, "user", 2), _tower(g, "item", 2)
    it_neg = _tower(g, "item", 2)
    u = ut.forward(g["user_features"])
    p = it.forward(g["pos_item_features"])
    nf = g["neg_item_features"]
    n = it_neg.forward(nf.reshape(-1, nf.shape[-1]))
    np.testing.assert_allclose(u, g["user_emb"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(p, g["pos_emb"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(n, g["neg_emb"], rtol=1e-5, atol=1e-6)
    ub, ib = float(g["user_bias"][0]), float(g["item_bias"][0])
    le, du_e, dp_e, dn_e, db = tt.explicit_loss(u, p, n, T, ub, ib, want_grad=True)
    li, du_i, dp_i = tt.in_batch_loss(u, p, T, want_grad=True)
    assert abs(le - float(g["explicit_loss"])) <= 1e-5 * abs(le)
    assert abs(li - float(g["inbatch_loss"])) <= 1e-5 * abs(li)
    assert abs(0.7 * le + 0.3 * li - float(g["loss"])) <= 1e-5 * float(g["loss"])
    assert abs(tt.mixed_loss(u, p, n, T, ub, ib) - float(g["loss"])) <= 1e-5 * float(g["loss"])
    du = 0.7 * du_e + 0.3 * du_i
    dp = 0.7 * dp_e + 0.3 * dp_i
    dn = 0.7 * dn_e
    np.testing.assert_allclose(du, g["grad.user_emb"], rtol=1e-4, atol=1e-7)
    np.testing.assert_allclose(dp, g["grad.pos_emb"], rtol=1e-4, atol=1e-7)
    np.testing.assert_allclose(dn, g["grad.neg_emb"], rtol=1e-4, atol=1e-7)
    np.testing.assert_allclose(0.7 * db, g["grad.user_bias"][0], rtol=1e-4, atol=1e-7)
    gu, _ = ut.backward(du)
    gp, _ = it.backward(dp)
    gn, _ = it_neg.backward(dn)
    for k, v in gu.items():
        ref = g["grad.user." + k]
        assert np.abs(v - ref).max() <= 2e-5 * max(np.abs(ref).max(), 1e-6), k
    for k in gp:
        ref = g["grad.item." + k]
        assert np.abs(gp[k] + gn[k] - ref).max() <= 2e-5 * max(np.abs(ref).max(), 1e-6), k


@pytest.mark.parametrize("name", ["step_ml1m", "step_small"])
def test_running_stats_and_eval_forward(golden_dir, name):
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    ut, it = _tower(g, "user", 2), _tower(g, "item", 2)
    ut.forward(g["user_features"], update_running=True)
    it.forward(g["pos_item_features"], update_running=True)
    nf = g["neg_item_features"]
    it.forward(nf.reshape(-1, nf.shape[-1]), update_running=True)  # second BN update in the same step
    for k in g.files:
        if k.startswith("after.") and "running" in k:
            tower, key = k[len("after."):].split(".", 1)
            got = (ut if tower == "user" else it).p[key]
            np.testing.assert_allclose(got, g[k], rtol=1e-5, atol=1e-6, err_msg=k)
    ue = ut.forward(g["user_features"], training=False)
    pe = it.forward(g["pos_item_features"], training=False)
    np.testing.assert_allclose(ue, g["user_emb_eval"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(pe, g["pos_emb_eval"], rtol=1e-5, atol=1e-6)
    li = tt.in_batch_loss(ue, pe, float(g["temperature"]))
    assert abs(li - float(g["inbatch_loss_eval"])) <= 1e-5 * abs(li)


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "cat_*.npz"))))
def test_categorical_towers_match_reference(path):
    g = np.load(path)
    act = str(g["activation"])
    ut, it = _tower(g, "user", 2, act), _tower(g, "item", 2, act)
    ucat = {k.split(".", 1)[1]: g[k] for k in g.files if k.startswith("user_cat.")}
    icat = {k.split(".", 1)[1]: g[k] for k in g.files if k.startswith("item_cat.")}
    u = ut.forward(g["user_num"], ucat)
    i = it.forward(g["item_num"], icat)
    np.testing.assert_allclose(u, g["user_emb"], rtol=2e-5, atol=2e-6)
    np.testing.assert_allclose(i, g["item_emb"], rtol=2e-5, atol=2e-6)
    T = float(g["temperature"])
    np.testing.assert_allclose((u * i).sum(-1) / T, g["similarity"], rtol=1e-4, atol=1e-5)
    loss, du, di = tt.in_batch_loss(u, i, T, want_grad=True)
    assert abs(loss - float(g["loss"])) <= 1e-5 * abs(loss)
    gu, _ = ut.backward(du)
    gi, _ = it.backward(di)
    for tower, grads in (("user", gu), ("item", gi)):
        for k, v in grads.items():
            ref = g[f"grad.{tower}.{k}"]
            assert np.abs(v - ref).max() <= 5e-5 * max(np.abs(ref).max(), 1e-6), (tower, k)
            if k.startswith("embeddings."):
                # gradient index set: exact (padding row 0 excluded)
                field = k.split(".")[1]
                idx = (ucat if tower == "user" else icat)[field]
                touched = tt.embedding_touched_rows(idx)
                assert np.array_equal(np.nonzero(np.abs(ref).sum(1))[0], touched) or \
                    set(np.nonzero(np.abs(ref).sum(1))[0]) <= set(touched.tolist())
                assert np.abs(v[0]).max() == 0


def test_kat_losses(golden_dir):
    g = np.load(os.path.join(golden_dir, "kat_losses.npz"))
    U = np.eye(4, 8)
    # closed forms (SURVEY §8c): -ln(e^10/(e^10+3)) and friends
    assert abs(tt.in_batch_loss(U, U, 0.1) - np.log1p(3 * np.exp(-10.0))) < 1e-9
    assert abs(tt.in_batch_loss(U, U, 0.1) - float(g["inbatch"])) < 1e-6
    assert abs(tt.explicit_loss(U, U, g["neg"], 0.1) - float(g["explicit"])) < 1e-6
    assert abs(tt.explicit_loss(U, U, g["neg"], 0.1, 0.5, 0.25) - float(g["explicit_bias"])) < 1e-6


# ---- exact inner-product top-K ------------------------------------------------------------------
def test_flat_ip_matches_reference_eval_twin():
    rng = np.random.default_rng(0)
    items = rng.standard_normal((3416, 128)).astype(np.float32)
    users = rng.standard_normal((64, 128)).astype(np.float32)
    flat_ip.normalize_L2(items); flat_ip.normalize_L2(users)
    train = {u: rng.choice(3416, size=rng.integers(0, 200), replace=False).tolist() for u in range(64)}
    twin = flat_ip.eval_twin_topk(users, items, train, list(range(64)), 100)
    idx = flat_ip.IndexFlatIP(128, db_block=1000)
    idx.add(items)
    D, I = idx.search(users, 100, exclude=[np.array(train[u], dtype=np.int64) for u in range(64)])
    for u in range(64):
        assert I[u].tolist() == twin[u]
    assert np.all(np.diff(D, axis=1) <= 0)


def test_flat_ip_semantics():
    rng = np.random.default_rng(1)
    x = rng.standard_normal((50, 16)).astype(np.float32)
    idx = flat_ip.IndexFlatIP(16)
    idx.add(x[:30]); idx.add(x[30:])
    assert idx.ntotal == 50
    q = rng.standard_normal((3, 16)).astype(np.float32)
    D, I = idx.search(q, 60)  # k > ntotal: padded with -1 / -FLT_MAX
    assert np.all(I[:, 50:] == -1) and np.all(D[:, 50:] == -flat_ip.FLT_MAX)
    full = q @ x.T
    for r in range(3):
        assert I[r, :50].tolist() == np.lexsort((np.arange(50), -full[r].astype(np.float64))).tolist()
    # ties: duplicated rows -> lower row id first
    xi = rng.integers(-4, 5, size=(5, 16)).astype(np.float32)  # exactly representable -> exact ties
    qi = rng.integers(-4, 5, size=(1, 16)).astype(np.float32)
    xd = np.concatenate([xi, xi], 0)
    idx2 = flat_ip.IndexFlatIP(16); idx2.add(xd)
    D2, I2 = idx2.search(qi, 4)
    best = int(np.lexsort((np.arange(5), -(qi[0] @ xi.T)))[0])
    assert I2[0, 0] == best and I2[0, 1] == best + 5 and D2[0, 0] == D2[0, 1]


def test_normalize_and_wrapper_semantics():
    x = np.array([[3.0, 4.0], [0.0, 0.0]], dtype=np.float32)
    flat_ip.normalize_L2(x)
    np.testing.assert_allclose(x, [[0.6, 0.8], [0.0, 0.0]], rtol=1e-6)
    fi = flat_ip.FaissIndexOracle({"dimension": 4})
    with pytest.raises(ValueError, match="Index not built yet"):
        fi.search(np.zeros((1, 4), np.float32))
    rng = np.random.default_rng(2)
    emb = rng.standard_normal((20, 4)).astype(np.float32)
    ids = [f"item_{i}" for i in range(20)]
    fi.build(emb, ids)
    got_ids, got_d = fi.search(emb[3], k=5)  # 1-D query promoted (retrieval.py:162-163)
    assert got_ids[0][0] == "item_3" and abs(got_d[0][0] - 1.0) < 1e-5 and len(got_ids[0]) == 5
    allow = ["item_1", "item_2", "item_3"]
    f_ids, _ = fi.search(emb[:2], k=2, filter_ids=allow)
    assert all(set(r) <= set(allow) for r in f_ids)
    fi.add(emb[:2] * 2.0, ["dup_a", "dup_b"])
    assert fi.current_size == 22 and fi.id_map[21] == "dup_b"


def test_bf16_round():
    import torch
    x = np.random.default_rng(3).standard_normal(4096).astype(np.float32)
    ref = torch.from_numpy(x).to(torch.bfloat16).to(torch.float32).numpy()
    assert np.array_equal(flat_ip.bf16_round(x), ref)


def test_feed_oracle_matches_reference_batches():
    """oracle/feed.py (sample_negative_items + __getitem__ + collate_fn restated) reproduces, bit for bit and from the
    same numpy seed, the batch the imported reference built (tests/golden/make_golden_feed.py)."""
    import os
    from oracle.feed import make_batch
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "feed_small.npz"))
    pos = {}
    for u, i in zip(g["in_user_idx"].tolist(), g["in_item_idx"].tolist()):
        pos.setdefault(u, []).append(i)
    np.random.seed(int(g["seed"]))
    b = make_batch(g["rows"].tolist(), g["in_user_idx"], g["in_item_idx"], g["in_label"], g["in_uf"], g["in_mf"], pos,
                   int(g["n_items"]), int(g["R"]), True)
    for k, v in b.items():
        ref = g["out_" + k]
        assert v.shape == ref.shape, k
        assert np.array_equal(v, ref), k
    # the sampler's contract, used as the property oracle for the device sampler
    for u, neg in zip(b["user_idx"].tolist(), b["neg_item_indices"].tolist()):
        assert len(set(neg)) == len(neg) and not (set(neg) & set(pos[u])) and all(0 <= x < int(g["n_items"]) for x in neg)


def test_wrapper_oracle_matches_the_reference_wrapper():
    """oracle.flat_ip.FaissIndexOracle (FaissIndex wrapper restated) against the REFERENCE's own FaissIndex /
    RetrievalEngine code run with a numpy stand-in for faiss (tests/golden/make_golden_wrapper.py): casts, 1-D promotion,
    cosine normalisation, id maps, the filter_ids post-pass with k_search = min(2k, N), incremental add."""
    import json
    import os
    from oracle.flat_ip import FaissIndexOracle
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "wrapper_small.npz"))
    cases = json.loads(str(g["cases_json"]))
    allowed = json.loads(str(g["allowed_json"]))
    emb, extra, qry, N, D = g["emb"], g["extra"], g["qry"], int(g["N"]), int(g["D"])
    ids = [f"item_{i}" for i in range(N)]
    extra_ids = [f"new_{i}" for i in range(len(extra))]

    def same(got, want):
        assert got[0] == want[0]                                   # item ids, list of lists
        assert len(got[1]) == len(want[1])
        for a, b in zip(got[1], want[1]):
            assert np.allclose(a, b, rtol=0, atol=1e-6)

    for metric in ("cosine", "ip"):
        ix = FaissIndexOracle({"dimension": D, "metric": metric})
        ix.build(emb.copy(), ids)
        same(ix.search(qry.copy(), k=10), cases[f"{metric}_k10"])
        same(ix.search(qry[0].copy(), k=5), cases[f"{metric}_1d_k5"])
        same(ix.search(qry.copy(), k=7, filter_ids=allowed), cases[f"{metric}_filter_k7"])
        ix.add(extra.copy(), extra_ids)
        same(ix.search(qry.copy(), k=10), cases[f"{metric}_after_add_k10"])
        assert ix.current_size == cases[f"{metric}_size"]
    ix = FaissIndexOracle({"dimension": D, "metric": "cosine"})
    ix.build(emb.copy(), ids)
    same(ix.search(qry[:2].copy(), k=6), cases["engine_retrieve_k6"])
    assert cases["engine_metrics_keys"] == ["avg_score", "cache_hit", "latency_ms", "num_results"]  # mirrored by b200rec.retrieval


def test_flat_ip_oracle_matches_the_reference_recommendation_twin():
    """IndexFlatIP restated (with the exclusion lists of the eval path) against the REFERENCE's generate_recommendations
    (scripts/evaluate_model.py:160-234: np.dot, -inf mask of the train items, argsort[::-1][:k]) on tie-free synthetic
    embeddings — the in-repo exact twin of the search the serving path delegates to faiss."""
    import os
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "evaltwin_small.npz"))
    items, users, test_users, k = g["items"], g["users"], g["test_users"], int(g["k"])
    train = {int(u): g["train_items"][g["train_indptr"][j]:g["train_indptr"][j + 1]]
             for j, u in enumerate(g["train_users"].tolist())}
    n_items = items.shape[0]
    excl = [np.unique(train[int(u)][train[int(u)] < n_items]).astype(np.int64) if int(u) in train
            else np.empty(0, np.int64) for u in test_users.tolist()]
    idx = flat_ip.IndexFlatIP(items.shape[1], db_block=500)
    idx.add(items)
    D, I = idx.search(users[test_users], k, exclude=excl)
    assert np.array_equal(I, g["recs"])
    twin = flat_ip.eval_twin_topk(users[test_users], items, {u: v.tolist() for u, v in train.items()}, test_users.tolist(), k)
    assert [twin[int(u)] for u in test_users.tolist()] == g["recs"].tolist()


def _metrics_cases():
    import json
    import os
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "metrics_small.npz"))
    cases = json.loads(str(g["cases_json"]))
    for c in cases.values():
        c["pred"] = {int(k): v for k, v in c["pred"].items()}
        c["gt"] = {int(k): set(v) for k, v in c["gt"].items()}
        c["exclude"] = {int(k): set(v) for k, v in c["exclude"].items()} if c["exclude"] else None
    return cases


def test_metrics_oracle_matches_the_reference_evaluator():
    """oracle/metrics.py (Evaluator.evaluate + per-user helpers restated) reproduces, number for number, what the
    imported reference computed (tests/golden/make_golden_metrics.py): distinct top-K lists, repeated ids, ragged lists,
    an exclusion dict, users without / with empty ground truth, ground-truth ids that are never recommended."""
    from oracle import metrics as M
    for name, c in _metrics_cases().items():
        got, mat = M.evaluate(c["pred"], c["gt"], c["k_values"], c["num_items"], c["exclude"])
        assert got.keys() == c["metrics"].keys()
        for k, v in c["metrics"].items():
            assert got[k] == v, (name, k, got[k], v)
        for j, k in enumerate(sorted(c["k_values"])):
            assert mat[:, 4 * j].tolist() == c["per_user_recall"][str(k)]
            assert mat[:, 4 * j + 2].tolist() == c["per_user_ndcg"][str(k)]


def test_blocked_baseline_search_equals_the_checker_on_tie_free_data():
    """oracle.flat_ip.search_blocked (threaded sgemm + topk, the CPU baseline's fallback without a C compiler) returns the same
    ids and scores as the deterministic checker IndexFlatIP.search when no two scores are equal."""
    rng = np.random.default_rng(8)
    cat = rng.standard_normal((5000, 24)).astype(np.float32)
    qry = rng.standard_normal((70, 24)).astype(np.float32)
    ix = flat_ip.IndexFlatIP(24)
    ix.add(cat)
    rD, rI = ix.search(qry, 30)
    D, I = flat_ip.search_blocked(cat, qry, 30, db_block=700, q_block=32)
    assert np.array_equal(I, rI) and np.allclose(D, rD, atol=1e-5)
    D, I = flat_ip.search_blocked(cat[:20], qry, 30)          # k > ntotal: -1 / -FLT_MAX padding
    assert (I[:, 20:] == -1).all() and (D[:, 20:] == -flat_ip.FLT_MAX).all()
    small = flat_ip.IndexFlatIP(24)
    small.add(cat[:20])
    assert np.array_equal(I[:, :20], small.search(qry, 30)[1][:, :20])


def test_flat_ip_oracle_agrees_with_an_independent_brute_force_library():
    """Third-party cross-check of the checker (faiss itself is not installable here): scikit-learn's brute-force
    NearestNeighbors under the cosine metric ranks unit-norm rows exactly as IndexFlatIP ranks them by inner product
    (cosine distance = 1 - ip), and torch.topk over the full fp32 score matrix gives the same lists."""
    neighbors = pytest.importorskip("sklearn.neighbors")
    rng = np.random.default_rng(21)
    cat = flat_ip.normalize_L2(rng.standard_normal((3000, 32)).astype(np.float32))
    qry = flat_ip.normalize_L2(rng.standard_normal((40, 32)).astype(np.float32))
    ix = flat_ip.IndexFlatIP(32, db_block=512)
    ix.add(cat)
    D, I = ix.search(qry, 25)
    nn = neighbors.NearestNeighbors(n_neighbors=25, algorithm="brute", metric="cosine").fit(cat.astype(np.float64))
    dist, ind = nn.kneighbors(qry.astype(np.float64))
    assert np.allclose(1.0 - dist, D, atol=1e-6)
    mism = I != ind                        # fp64 vs fp32 scores may swap neighbours closer than fp32 resolution
    assert mism.mean() < 0.02 and (np.abs((1.0 - dist) - D)[mism] < 1e-6).all()
    import torch
    ts, ti = torch.topk(torch.from_numpy(qry) @ torch.from_numpy(cat).T, 25, dim=1)
    m2 = I != ti.numpy()
    assert np.allclose(D, ts.numpy(), atol=1e-6) and m2.mean() < 0.02


def test_reservoir_baseline_search_equals_the_checker_including_ties():
    """oracle.flat_ip.search_reservoir (blocked sgemm + the C reservoir result handler of oracle/csrc/flat_select.c: what
    bench.py times as the CPU baseline) returns exactly the checker's lists, also when scores tie (duplicated rows: the
    order is score desc, row asc, and only a strictly greater score displaces the k-th), for ragged block shapes, for
    k larger than the catalogue and when reservoirs overflow many times (rows sorted by increasing score)."""
    rng = np.random.default_rng(9)
    cat = rng.standard_normal((6000, 24)).astype(np.float32)
    cat[1000:1500] = cat[:500]            # exact score ties between rows r and r + 1000
    cat[5990:] = cat[10:20]
    qry = rng.standard_normal((70, 24)).astype(np.float32)
    ix = flat_ip.IndexFlatIP(24)
    ix.add(cat)
    for k in (1, 30, 100):
        rD, rI = ix.search(qry, k)
        for db_block, q_block, threads in ((700, 32, 3), (4096, 1024, 0), (64, 7, 2)):
            D, I = flat_ip.search_reservoir(cat, qry, k, threads, db_block=db_block, q_block=q_block)
            assert np.array_equal(I, rI), (k, db_block)
            assert np.allclose(D, rD, atol=1e-5)
    D, I = flat_ip.search_reservoir(cat[:20], qry, 30)        # k > ntotal: -1 / -FLT_MAX padding
    assert (I[:, 20:] == -1).all() and (D[:, 20:] == -flat_ip.FLT_MAX).all()
    small = flat_ip.IndexFlatIP(24)
    small.add(cat[:20])
    assert np.array_equal(I[:, :20], small.search(qry, 30)[1][:, :20])
    # worst case for the reservoir: every row beats the threshold (rows ordered by increasing score for every query)
    base = np.abs(rng.standard_normal((1, 8))).astype(np.float32)
    ramp = (np.arange(1, 3001, dtype=np.float32)[:, None] * base)
    qpos = np.abs(rng.standard_normal((5, 8))).astype(np.float32)
    ix2 = flat_ip.IndexFlatIP(8)
    ix2.add(ramp)
    rD, rI = ix2.search(qpos, 10)
    D, I = flat_ip.search_reservoir(ramp, qpos, 10, 2, db_block=256)
    assert np.array_equal(I, rI) and np.allclose(D, rD, rtol=1e-6)
    # and it agrees with the torch.topk variant on tie-free data
    cat3 = rng.standard_normal((5000, 24)).astype(np.float32)
    assert np.array_equal(flat_ip.search_reservoir(cat3, qry, 30)[1], flat_ip.search_blocked(cat3, qry, 30)[1])


def test_round2_goldens_are_consistent(golden_dir):
    """content_branch.npz / trajectory_120.npz (tests/golden/make_golden_round2.py, imported reference): the trajectory's
    batches regenerate bit for bit from the stored seed on this machine (torch CPU generator), the reference's loss
    falls from ~ln-scale to < 2 over the 120 steps, the content-branch embeddings are unit rows."""
    import os
    import sys
    import numpy as np
    sys.path.insert(0, golden_dir)
    from trajectory_batches import make_batches
    g = np.load(os.path.join(golden_dir, "trajectory_120.npz"))
    batches = make_batches(int(g["seed"]), int(g["steps"]), int(g["B"]), int(g["R"]), int(g["user_dim"]), int(g["item_dim"]))
    sums = [float(b["user_features"].double().sum() + b["pos_item_features"].double().sum()
                  + b["neg_item_features"].double().sum()) for b in batches]
    assert np.array_equal(np.asarray(sums), g["batch_checksum"])
    assert g["losses"].shape == (120,) and g["losses"][0] > 5.0 and g["losses"][-1] < 2.0
    assert abs(g["losses"].mean() - float(g["epoch_mean"])) < 1e-6
    c = np.load(os.path.join(golden_dir, "content_branch.npz"))
    for k in ("emb_train", "emb_eval"):
        assert np.allclose(np.linalg.norm(c[k], axis=1), 1.0, atol=1e-5)
    assert any(k.startswith("grad.content_projection") for k in c.files)


def test_oracle_content_projection_branch_matches_reference(golden_dir):
    """oracle.TowerOracle with the ItemTower content branch (two_tower.py:184-191,264-266) against the golden generated
    from the imported reference: train-mode (batch statistics) and eval-mode embeddings, and the gradient of
    sum(emb * w) with respect to every parameter."""
    import os
    import numpy as np
    from oracle.two_tower import TowerOracle
    g = np.load(os.path.join(golden_dir, "content_branch.npz"))
    t = TowerOracle({k[3:]: g[k] for k in g.files if k.startswith("sd.")}, 2, "relu")
    # the golden's eval forward ran after the training forward had updated the running statistics
    for training, key in ((True, "emb_train"), (False, "emb_eval")):
        e = t.forward(g["numerical"], {"genre": g["genre"]}, training=training, content=g["content"],
                      update_running=training)
        assert np.abs(e - g[key]).max() <= 2e-6, key
        if training:
            # gradient of sum(emb * w) w.r.t. every parameter, the content_projection Linears and the table included
            grads, _ = t.backward(g["w"])
            want = {k[5:]: g[k] for k in g.files if k.startswith("grad.")}
            assert set(grads) == set(want)
            for k, ref in want.items():
                assert np.abs(grads[k] - ref).max() <= 2e-5 * max(np.abs(ref).max(), 1e-6), k


# a checkout of the original project (the reference the goldens were generated from), e.g. REFERENCE_ROOT=../upstream
REFERENCE_ROOT = os.environ.get("REFERENCE_ROOT", "")
needs_reference = pytest.mark.skipif(not (REFERENCE_ROOT and os.path.isdir(os.path.join(REFERENCE_ROOT, "src"))),
                                     reason="set REFERENCE_ROOT to a checkout of the original project")


@needs_reference
def test_committed_goldens_regenerate_from_the_imported_reference(tmp_path):
    """Provenance of tests/golden/*.npz: every generator script is re-run here (each imports the unmodified reference and
    runs it on seeded inputs) and what it writes must equal the committed fixture — identical integer / string arrays,
    floating-point arrays bit-identical at the generating thread count and within 1e-4 of the array's scale otherwise
    (tests/golden/verify_goldens.py states the one exception, the chaotic 120-step trajectory)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("verify_goldens", os.path.join(os.path.dirname(__file__), "golden",
                                                                                "verify_goldens.py"))
    vg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(vg)
    vg.regenerate(str(tmp_path))
    committed, problems, worst = vg.compare(str(tmp_path))
    assert len(committed) >= 14
    assert not problems, problems[:10]


@needs_reference
@pytest.mark.parametrize("seed", range(6))
def test_oracle_matches_the_live_reference_on_random_configurations(seed):
    """Beyond the stored fixtures: the numpy restatement against the IMPORTED reference itself (torch-CPU autograd) on
    configurations drawn at random — depth 1-3, every activation, ragged widths, 0-3 categorical fields per tower with
    small and large cardinalities (row width min(50, (card+1)//2), padding id 0 present in the batch), batch sizes down
    to 2, explicit / in-batch / mixed loss with random biases and temperature: embeddings, losses, every parameter
    gradient (tables included) and the BatchNorm running statistics after the step."""
    import sys
    import torch
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    from src.models.two_tower import ItemTower, TwoTowerModel, UserTower
    rng = np.random.default_rng(1000 + seed)
    torch.manual_seed(1000 + seed)
    act = ["relu", "gelu", "leaky_relu", "tanh", "sigmoid", "relu"][seed]
    L = int(rng.integers(1, 4))
    hidden = [int(rng.integers(3, 40)) for _ in range(L)]
    E = int(rng.integers(2, 33))
    B = int([2, 5, 33, 64, 17, 128][seed])
    R = int(rng.integers(2, 6))               # neg_ratio 1 crashes in the reference (SURVEY section 7.8)
    ud, idim = int(rng.integers(1, 12)), int(rng.integers(1, 24))
    ucards = {f"uf{j}": int(rng.choice([1, 2, 7, 40, 300])) for j in range(int(rng.integers(0, 4)))}
    icards = {f"if{j}": int(rng.choice([1, 3, 9, 120, 99])) for j in range(int(rng.integers(0, 4)))}
    ut = UserTower(ud, E, hidden, 0.0, act, ucards or None)
    it = ItemTower(idim, E, hidden, 0.0, act, icards or None, use_content_embedding=False)
    T = float(rng.uniform(0.03, 0.5))
    model = TwoTowerModel(ut, it, temperature=T, use_bias=True)
    with torch.no_grad():
        model.user_bias.fill_(float(rng.normal(0, 0.3)))
        model.item_bias.fill_(float(rng.normal(0, 0.3)))
        for m in model.modules():
            if isinstance(m, torch.nn.BatchNorm1d):
                m.weight.copy_(1.0 + 0.2 * torch.randn(m.weight.shape))
                m.bias.copy_(0.1 * torch.randn(m.bias.shape))
    model.train()
    sd_u = {k: v.detach().numpy().copy() for k, v in ut.state_dict().items()}
    sd_i = {k: v.detach().numpy().copy() for k, v in it.state_dict().items()}
    uf = rng.standard_normal((B, ud)).astype(np.float32)
    pf = rng.standard_normal((B, idim)).astype(np.float32)
    nf = rng.standard_normal((B * R, idim)).astype(np.float32)
    ucat = {k: rng.integers(0, c + 1, size=B) for k, c in ucards.items()}       # 0 = padding id
    icat = {k: rng.integers(0, c + 1, size=B) for k, c in icards.items()}
    ncat = {k: rng.integers(0, c + 1, size=B * R) for k, c in icards.items()}
    t = lambda d: {k: torch.from_numpy(v) for k, v in d.items()}
    u = model.get_user_embeddings({"numerical": torch.from_numpy(uf), "categorical": t(ucat)})
    p = model.get_item_embeddings({"numerical": torch.from_numpy(pf), "categorical": t(icat)})
    n = model.get_item_embeddings({"numerical": torch.from_numpy(nf), "categorical": t(ncat)})
    le_ref, li_ref = model.contrastive_loss(u, p, n), model.in_batch_negative_loss(u, p)
    mode = seed % 3
    loss_ref = [0.7 * le_ref + 0.3 * li_ref, li_ref, le_ref][mode]
    loss_ref.backward()
    # ---- the oracle on the same numbers
    uo, po, no = tt.TowerOracle(sd_u, L, act), tt.TowerOracle(sd_i, L, act), tt.TowerOracle(sd_i, L, act)
    ue, pe = uo.forward(uf, ucat), po.forward(pf, icat)
    ne = no.forward(nf, ncat)
    np.testing.assert_allclose(ue, u.detach().numpy(), rtol=2e-5, atol=2e-6)
    np.testing.assert_allclose(pe, p.detach().numpy(), rtol=2e-5, atol=2e-6)
    np.testing.assert_allclose(ne, n.detach().numpy(), rtol=2e-5, atol=2e-6)
    ub, ib = float(model.user_bias.item()), float(model.item_bias.item())
    le, du_e, dp_e, dn_e, db = tt.explicit_loss(ue, pe, ne, T, ub, ib, want_grad=True)
    li, du_i, dp_i = tt.in_batch_loss(ue, pe, T, want_grad=True)
    assert abs(le - le_ref.item()) <= 2e-5 * max(abs(le), 1e-3) and abs(li - li_ref.item()) <= 2e-5 * max(abs(li), 1e-3)
    we, wi = [(0.7, 0.3), (0.0, 1.0), (1.0, 0.0)][mode]
    gu, _ = uo.backward(we * du_e + wi * du_i)
    gp, _ = po.backward(we * dp_e + wi * dp_i)
    gn, _ = no.backward(we * dn_e)
    if we:
        assert abs(we * db - float(model.user_bias.grad)) <= 1e-4 * max(abs(we * db), 1e-4)
    for tower, grads, extra in ((ut, gu, None), (it, gp, gn)):
        named = dict(tower.named_parameters())
        for k, v in grads.items():
            ref = named[k].grad
            ref = np.zeros_like(v) if ref is None else ref.numpy()
            got = v + (extra[k] if extra is not None and we else 0)
            # fp64 oracle vs the reference's fp32 autograd: 1e-4 of the gradient's scale, 5e-4 for the 2- and 5-sample
            # batches (BatchNorm over a handful of rows divides by a variance that fp32 itself resolves poorly)
            tol = 1e-4 if B >= 16 else 5e-4
            assert np.abs(got - ref).max() <= tol * max(np.abs(ref).max(), 1e-5), (k, act, L)
            if k.startswith("embeddings."):
                assert np.abs(got[0]).max() == 0                     # padding row: no gradient
    # BatchNorm running statistics after the three tower passes of the step (item tower: two updates)
    uo.forward(uf, ucat, update_running=True)
    po.forward(pf, icat, update_running=True)
    po.forward(nf, ncat, update_running=True)
    for tower, orc in ((ut, uo), (it, po)):
        for k, v in tower.state_dict().items():
            if "running" in k:
                np.testing.assert_allclose(orc.p[k], v.numpy(), rtol=1e-4, atol=1e-6, err_msg=k)
