"""CPU-side checks (no GPU): the C-ABI library loads and exports every symbol include/b200rec.h declares, the ctypes
binding agrees with the header, the drop-in modules keep the reference's state-dict layout, the product has no CPU
fallback, and the multi-rank retrieval plumbing (world_size 2, gloo) reproduces the single-process oracle."""
import os
import re
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_decls():
    hdr = open(os.path.join(ROOT, "include", "b200rec.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    return re.findall(r"\b(b200rec_\w+)\s*\(([^;]*?)\)\s*;", hdr)


def test_library_builds_and_exports_every_declared_symbol():
    import __graft_entry__ as g
    g.build()
    from b200rec import _native
    lib = _native.lib()
    decls = _header_decls()
    assert len(decls) >= 30
    for name, args in decls:
        assert hasattr(lib, name), f"{name} declared in include/b200rec.h but not exported"
        nargs = 0 if args.strip() in ("void", "") else len(args.split(","))
        assert name in _native.SIGNATURES, f"{name} has no ctypes signature"
        assert len(_native.SIGNATURES[name][1]) == nargs, f"{name}: binding has {len(_native.SIGNATURES[name][1])} args, header {nargs}"
    assert lib.b200rec_version() == 1
    assert lib.b200rec_launch_count() == 0  # nothing has been launched: no compute without a GPU


def test_library_is_sm100a_only_and_its_hot_kernels_are_tcgen05_tma_tmem():
    """No GPU needed: the fat binary holds sm_100a cubins only (no PTX for another target, no second architecture), and
    the SASS of the kernels on the hot path carries the Blackwell-native instructions DESIGN.md claims for them —
    UTCHMMA(.2CTA) = tcgen05.mma (cta_group::2), UTMALDG = TMA tensor loads, LDTM / STTM = tcgen05.ld / .st (TMEM)."""
    import shutil
    import subprocess
    from b200rec import _native
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    elfs = subprocess.run([cuobjdump, "-lelf", _native.LIB_PATH], capture_output=True, text=True).stdout.split("\n")
    archs = {m.group(1) for m in (re.search(r"\.(sm_\w+)\.cubin", e) for e in elfs) if m}
    assert archs == {"sm_100a"}, archs
    ptx = subprocess.run([cuobjdump, "-lptx", _native.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_" not in ptx or set(re.findall(r"sm_\w+", ptx)) <= {"sm_100a"}
    sass = subprocess.run([cuobjdump, "-sass", _native.LIB_PATH], capture_output=True, text=True).stdout
    per_kernel, cur = {}, None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = per_kernel.setdefault(m.group(1), {})
            continue
        m = re.search(r"/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", line)
        if m and cur is not None:
            for op in ("UTCHMMA.2CTA", "UTCHMMA", "UTMALDG", "LDTM", "STTM"):
                if m.group(1).startswith(op):
                    cur[op] = cur.get(op, 0) + 1
                    break

    def kernels(*parts):
        hit = [c for name, c in per_kernel.items() if all(p in name for p in parts)]
        assert hit, f"no kernel matching {parts}"
        return hit

    # K4 headline kernel: CTA pairs, TMA-fed, TMEM accumulators read back by the select epilogue
    for c in kernels("stream_scores2_kernel", "ILi2E", "TopkEpiTILb0E"):   # release instantiation (no debug stamps)
        assert c.get("UTCHMMA.2CTA", 0) > 0 and c.get("UTMALDG", 0) > 0 and c.get("LDTM", 0) > 0, c
    # K3: LSE forward and the flash-style backward (G written to TMEM with tcgen05.st = STTM)
    for c in kernels("stream_scores_kernel", "LseEpi"):
        assert c.get("UTCHMMA", 0) > 0 and c.get("UTMALDG", 0) > 0 and c.get("LDTM", 0) > 0, c
    for c in kernels("inbatch_grad_kernel"):
        assert c.get("UTCHMMA", 0) > 0 and c.get("UTMALDG", 0) > 0 and c.get("LDTM", 0) > 0 and c.get("STTM", 0) > 0, c
    # K2 fused MLP layers and the generic tile GEMM
    for c in kernels("mlp_fused_kernel") + kernels("gemm_bf16_tn_kernel"):
        assert c.get("UTCHMMA", 0) > 0 and c.get("LDTM", 0) > 0, c


def test_argument_errors_are_reported_without_a_gpu():
    from b200rec import _native
    lib = _native.lib()
    assert lib.b200rec_topk_workspace_bytes(0, 128, 4, 10) == 0
    assert "empty" in _native.last_error()
    assert lib.b200rec_topk_workspace_bytes(1000, 100, 4, 10) == 0
    assert "multiple of 64" in _native.last_error()
    assert lib.b200rec_topk_merge(None, None, 1, 1, 1, 1, 0, 0, None, None, None) != 0
    assert "null" in _native.last_error()


def test_every_entry_point_rejects_null_arguments_with_a_message():
    """Error behaviour of the whole C-ABI, no GPU needed: called with null pointers and zero sizes every int-returning
    entry point that takes a pointer returns non-zero and explains itself through b200rec_last_error() — no crash, no
    launch, no exception across the ABI (the two pure shape predicates return 0 = "no")."""
    import ctypes as C
    from b200rec import _native
    lib = _native.lib()
    predicates = {"b200rec_topk_has_sample", "b200rec_inbatch_grad_supported"}
    before = lib.b200rec_launch_count()
    checked = 0
    for name, (restype, argtypes) in _native.SIGNATURES.items():
        if restype is not C.c_int or C.c_void_p not in argtypes and name not in predicates:
            continue
        args = [None if t is C.c_void_p else (0.0 if t in (C.c_float, C.c_double) else 0) for t in argtypes]
        rc = getattr(lib, name)(*args)
        if name in predicates:
            assert rc == 0, name
            continue
        assert rc != 0, f"{name} accepted null pointers"
        msg = _native.last_error()
        assert msg and ("null" in msg or "empty" in msg or "must" in msg), f"{name}: unhelpful error {msg!r}"
        checked += 1
    assert checked >= 45
    assert lib.b200rec_launch_count() == before


def test_header_is_plain_c_and_a_c_host_links(tmp_path):
    """The boundary is a C ABI, not a Python extension: include/b200rec.h compiles as pedantic C99, a C program links
    against libb200rec.so and gets its errors as return codes + b200rec_last_error() (tests/c_host/host.c)."""
    import shutil
    import subprocess
    from b200rec import _native
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no gcc")
    libdir = os.path.dirname(_native.LIB_PATH)
    exe = str(tmp_path / "host")
    r = subprocess.run([gcc, "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "tests", "c_host", "host.c"), "-o", exe, "-L", libdir, "-lb200rec",
                        f"-Wl,-rpath,{libdir}"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0, (r.returncode, r.stdout, r.stderr)
    assert "config-3 workspace" in r.stdout


def test_no_cpu_fallback():
    from b200rec.training_utils import create_two_tower_model_for_training
    m = create_two_tower_model_for_training(3, 20)
    m.eval()
    with pytest.raises(RuntimeError, match="no CPU path"):
        m.get_user_embeddings({"numerical": torch.randn(4, 3)})
    with pytest.raises(RuntimeError, match="no CPU path"):
        m.in_batch_negative_loss(torch.randn(4, 8), torch.randn(4, 8))
    if not torch.cuda.is_available():
        from b200rec.retrieval import FlatIPDeviceIndex
        with pytest.raises(RuntimeError, match="no CPU search path"):
            FlatIPDeviceIndex(16)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "real-time-recommendation-system-with-feature-store_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b|\boracle\.\w+\(|oracle/", src, flags=re.M), \
                    f"{f} imports or calls the oracle"


def test_state_dict_layout_and_param_counts():
    from b200rec.training_utils import count_parameters, create_two_tower_model_for_training
    # the two parameter counts the reference publishes (results/EVALUATION_REPORT.md:63)
    final = create_two_tower_model_for_training(3, 20, {"embedding_dim": 128, "hidden_layers": [256, 128]})
    before = create_two_tower_model_for_training(3, 20, {"embedding_dim": 64, "hidden_layers": [128, 64]})
    assert count_parameters(final) == 106754
    assert count_parameters(before) == 28802
    keys = list(final.user_tower.state_dict().keys())
    assert keys[:3] == ["mlp.0.weight", "mlp.0.bias", "mlp.2.weight"]
    assert "mlp.2.running_var" in keys and "mlp.2.num_batches_tracked" in keys and "mlp.8.weight" in keys
    assert final.user_tower.mlp[0].weight.shape == (256, 3)  # [out, in] Linear layout


def _golden_state(name, prefix):
    """(keys in order, {key: array}) of the state dict stored under `prefix.` in tests/golden/<name>.npz."""
    g = np.load(os.path.join(ROOT, "tests", "golden", name + ".npz"))
    keys = [k[len(prefix) + 1:] for k in g.files if k.startswith(prefix + ".")]
    return keys, {k: g[prefix + "." + k] for k in keys}


def _assert_same_state(module, golden, prefix, skip=lambda k: False):
    keys, want = _golden_state(golden, prefix)
    sd = module.state_dict()
    assert list(sd.keys()) == keys, (golden, prefix)
    for k in keys:
        if not skip(k):
            assert np.array_equal(sd[k].detach().cpu().numpy(), want[k]), (golden, prefix, k)


def _overwritten_after_init(k):
    """Entries the golden generators change after construction (tests/golden/make_golden.py randomize_bn: BatchNorm
    affine parameters and Linear biases from a separate generator; the stored running statistics are post-forward)."""
    return not (k.endswith(".weight") and (k.startswith("embeddings.") or k.split(".")[1] in ("0", "4", "8")))


def test_same_init_and_keys_as_the_imported_reference():
    """Same RNG consumption order as the reference => identical initial weights: the reference's factory built towers
    with categorical tables (cat_*.npz) and an ItemTower with the content branch (content_branch.npz) from a seed; the
    same seed here gives the same state-dict keys, layouts and initial Linear weights / embedding tables, bit for bit."""
    from b200rec.two_tower import ItemTower, create_two_tower_model
    for act in ("relu", "gelu"):
        cfg = {"embedding_dim": 32, "temperature": 0.1,
               "user_tower": {"input_dim": 10, "hidden_layers": [64, 32], "dropout_rate": 0.0, "activation": act,
                              "categorical_features": {"category": 10, "subcategory": 5}},
               "item_tower": {"input_dim": 15, "hidden_layers": [64, 32], "dropout_rate": 0.0, "activation": act,
                              "categorical_features": {"genre": 30, "studio": 200}, "use_content_embedding": False}}
        torch.manual_seed(20)
        ours = create_two_tower_model(cfg)
        _assert_same_state(ours.user_tower, f"cat_{act}", "user", _overwritten_after_init)
        _assert_same_state(ours.item_tower, f"cat_{act}", "item", _overwritten_after_init)
        assert ours.temperature == 0.1
    torch.manual_seed(41)
    it = ItemTower(input_dim=12, embedding_dim=32, hidden_layers=[64, 48], dropout_rate=0.0, activation="relu",
                   categorical_features={"genre": 20}, use_content_embedding=True, content_embedding_dim=64)
    _assert_same_state(it, "content_branch", "sd", lambda k: k.startswith("mlp.") and k.split(".")[1] in ("2", "6"))


def test_checkpoints_are_interchangeable_with_the_reference(tmp_path):
    """save_model / load_model in both directions (reference two_tower.py:516-546): a checkpoint in the reference's
    layout holding the reference's own initial state (trajectory_120.npz) loads into b200rec, and what b200rec writes
    has that layout — the same file keys, state-dict keys and tensors, biases and temperature."""
    from b200rec.two_tower import create_two_tower_model
    keys, ref = _golden_state("trajectory_120", "sd")
    tower = lambda t: {k[len(t) + 1:]: torch.from_numpy(ref[k].copy()) for k in keys if k.startswith(t + ".")}
    cfg = {"embedding_dim": 64, "temperature": 0.05,
           "user_tower": {"input_dim": 3, "hidden_layers": [128, 64]},
           "item_tower": {"input_dim": 20, "hidden_layers": [128, 64], "use_content_embedding": False}}
    path = str(tmp_path / "reference_layout.pth")
    torch.save({"user_tower_state": tower("user_tower"), "item_tower_state": tower("item_tower"), "temperature": 0.123,
                "user_bias": torch.nn.Parameter(torch.tensor([0.25])),
                "item_bias": torch.nn.Parameter(torch.tensor([-0.5]))}, path)
    torch.manual_seed(99)
    ours = create_two_tower_model(cfg)
    ours.load_model(path)
    _assert_same_state(ours.user_tower, "trajectory_120", "sd.user_tower")
    _assert_same_state(ours.item_tower, "trajectory_120", "sd.item_tower")
    assert ours.temperature == 0.123
    assert ours.user_bias.item() == 0.25 and ours.item_bias.item() == -0.5
    path2 = str(tmp_path / "ours.pth")
    ours.save_model(path2)
    ck = torch.load(path2, map_location="cpu", weights_only=False)
    assert sorted(ck.keys()) == ["item_bias", "item_tower_state", "temperature", "user_bias", "user_tower_state"]
    for t in ("user_tower", "item_tower"):
        want = tower(t)
        assert list(ck[t + "_state"].keys()) == list(want.keys())
        for k, v in want.items():
            assert torch.equal(ck[t + "_state"][k], v), (t, k)
    assert ck["temperature"] == 0.123 and ck["user_bias"].item() == 0.25 and ck["item_bias"].item() == -0.5


# golden -> (seed, user_dim, item_dim, config) the reference's create_two_tower_model_for_training was called with
# (tests/golden/make_golden.py, make_golden_round2.py)
_FACTORY_GOLDENS = {
    "trajectory_120": (77, 3, 20, {"embedding_dim": 64, "hidden_layers": [128, 64], "dropout_rate": 0.0,
                                   "temperature": 0.05}),
    "step_ml1m": (11, 3, 20, {"embedding_dim": 128, "hidden_layers": [256, 128], "dropout_rate": 0.0,
                              "temperature": 0.05}),
    "step_small": (12, 6, 9, {"embedding_dim": 64, "hidden_layers": [128, 64], "dropout_rate": 0.0, "temperature": 0.1}),
}


@pytest.mark.parametrize("golden", sorted(_FACTORY_GOLDENS))
def test_training_factory_matches_the_reference(golden):
    """create_two_tower_model_for_training (reference src/training/utils.py:14-71) against what the reference's factory
    built from the same seed: same RNG consumption (bit-identical initial weights: the whole state dict where the
    generator stored it untouched, the Linear weights otherwise), same keys, temperature and parameter count."""
    from b200rec.training_utils import count_parameters, create_two_tower_model_for_training
    seed, ud, idim, cfg = _FACTORY_GOLDENS[golden]
    torch.manual_seed(seed)
    ours = create_two_tower_model_for_training(ud, idim, cfg)
    if golden == "trajectory_120":
        _assert_same_state(ours, golden, "sd")
        user = _golden_state(golden, "sd.user_tower")[1]
        item = _golden_state(golden, "sd.item_tower")[1]
        temperature = cfg["temperature"]
    else:
        _assert_same_state(ours.user_tower, golden, "user", _overwritten_after_init)
        _assert_same_state(ours.item_tower, golden, "item", _overwritten_after_init)
        user, item = _golden_state(golden, "user")[1], _golden_state(golden, "item")[1]
        temperature = float(np.load(os.path.join(ROOT, "tests", "golden", golden + ".npz"))["temperature"])
    assert np.float32(ours.temperature) == np.float32(temperature)
    learnable = sum(v.size for t in (user, item) for k, v in t.items() if "running" not in k and "num_batches" not in k)
    assert count_parameters(ours) == learnable + 2      # + user_bias, item_bias
    assert [x.p for x in ours.modules() if isinstance(x, torch.nn.Dropout)] == [cfg["dropout_rate"]] * 4


def test_shard_bounds_cover_the_catalogue():
    from b200rec.dist import shard_bounds
    for n, w in ((10_000_000, 8), (1001, 4), (7, 8), (5, 1)):
        spans = [shard_bounds(n, w, r) for r in range(w)]
        assert spans[0][0] == 0 and spans[-1][1] == n
        assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
        assert max(h - l for l, h in spans) - min(h - l for l, h in spans) <= 1


def _gloo_worker(rank, world, port, tmp):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    from b200rec.dist import ShardedFlatIndex, shard_bounds
    from oracle.flat_ip import IndexFlatIP, merge_topk
    dist.init_process_group("gloo", rank=rank, world_size=world)
    rng = np.random.default_rng(5)
    N, Q, D, k = 5003, 37, 16, 25
    cat = rng.standard_normal((N, D)).astype(np.float32)
    cat[100:140] = cat[4000:4040]  # ties across shards
    qry = rng.standard_normal((Q, D)).astype(np.float32)
    lo, hi = shard_bounds(N, world, rank)
    ix = IndexFlatIP(D)
    ix.add(cat[lo:hi])

    def local(q, kk, tau=None):  # the oracle stands in for the CUDA kernel: same contract, global ids via the offset
        s, i = ix.search(q, kk)
        i = np.where(i >= 0, i + lo, -1)
        if tau is not None:  # shared thresholds: a shard drops what cannot reach the global top-k
            drop = s < tau.numpy()[:, None]
            s, i = np.where(drop, -np.finfo(np.float32).max, s), np.where(drop, -1, i)
        return torch.from_numpy(s.astype(np.float32)), torch.from_numpy(i)

    def sample(q, kk):  # any k distinct local rows per query: here the best of the first 400 rows of the shard
        sub = IndexFlatIP(D)
        sub.add(cat[lo:lo + 400])
        return torch.from_numpy(sub.search(q, kk)[0])

    def merge(s, i, kk):
        ms, mi = merge_topk([s[p].numpy() for p in range(s.shape[0])], [i[p].numpy() for p in range(i.shape[0])], kk)
        return torch.from_numpy(ms), torch.from_numpy(mi)

    s, i = ShardedFlatIndex(local, merge, local_sample=sample).search(qry, k)
    full = IndexFlatIP(D)
    full.add(cat)
    rs, ri = full.search(qry, k)
    ok = np.array_equal(i.numpy(), ri) and np.allclose(s.numpy(), rs, atol=1e-6)
    with open(os.path.join(tmp, f"ok{rank}"), "w") as fh:
        fh.write("1" if ok else "0")
    dist.destroy_process_group()


def test_sharded_retrieval_world_size_2_gloo(tmp_path):
    import torch.multiprocessing as mp
    port = 29500 + (os.getpid() % 2000)
    mp.spawn(_gloo_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert [open(tmp_path / f"ok{r}").read() for r in range(2)] == ["1", "1"]


def test_retrieval_batcher_groups_concurrent_requests():
    """Host logic of the serving micro-batcher (no GPU: a stand-in model and index): concurrent requests share one tower
    forward and one search, every caller gets its own rows cut to its own k, failures reach every waiting caller."""
    import asyncio
    import torch
    from b200rec.serving import RetrievalBatcher

    class Model:
        def __init__(self):
            self.w = torch.nn.Parameter(torch.eye(4))
            self.calls = []

        def parameters(self):
            return iter([self.w])

        def get_user_embeddings(self, feats):
            self.calls.append(tuple(feats["numerical"].shape))
            return feats["numerical"] @ self.w

    class Index:
        def __init__(self):
            self.calls = []
            self.fail = False

        def search(self, emb, k):
            if self.fail:
                raise ValueError("Index not built yet")
            self.calls.append((emb.shape[0], k))
            return ([[f"item_{int(e[0])}_{j}" for j in range(k)] for e in emb],
                    [[float(e[0]) - j for j in range(k)] for e in emb])

    class Engine:
        def __init__(self):
            self.index, self.total_queries, self.total_latency = Index(), 0, 0.0

        def account(self, seconds, calls=1):                      # RetrievalEngine's bookkeeping contract (seconds)
            self.total_queries += calls
            self.total_latency += seconds

    async def run():
        model, engine = Model(), Engine()
        b = RetrievalBatcher(model, engine, max_batch=4, max_wait_ms=5.0)
        reqs = [({"numerical": torch.tensor([[float(i), 0., 0., 0.]]), "categorical": {}}, 2 + i % 3) for i in range(10)]
        out = await asyncio.gather(*[b.recommend(f, k) for f, k in reqs])
        assert [c[0] for c in model.calls] == [4, 4, 2] and [c[0] for c in engine.index.calls] == [4, 4, 2]
        assert engine.index.calls[0][1] == 4                      # searched with the largest k of the batch
        for i, ((ids, scores, m), (_, k)) in enumerate(zip(out, reqs)):
            assert ids == [[f"item_{i}_{j}" for j in range(k)]] and len(scores[0]) == k and m["num_results"] == k
        assert engine.total_queries == 10 and b.batches == 3
        # per-request latency in SECONDS: every request is charged the shared search it waited for
        assert abs(engine.total_latency - sum(m["latency_ms"] for _, _, m in out) / 1e3) < 1e-9
        engine.index.fail = True
        res = await asyncio.gather(*[b.recommend(f, k) for f, k in reqs[:3]], return_exceptions=True)
        assert all(isinstance(r, ValueError) for r in res)

    asyncio.run(run())


def _gloo_dp_worker(rank, world, port, tmp):
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    sys.path.insert(0, ROOT)
    from b200rec.dist import DataParallel, ShardedFlatIndex, _AllGatherRows
    dist.init_process_group("gloo", rank=rank, world_size=world)
    g = torch.Generator().manual_seed(3)
    B, E = 5, 4
    xs = [torch.randn(B, E, generator=g) for _ in range(world)]          # every rank's local rows (same on all ranks)
    ws = [torch.randn(world * B, E, generator=g) for _ in range(world)]  # every rank's weights on the gathered rows
    x = xs[rank].clone().requires_grad_(True)
    y = _AllGatherRows.apply(x, None)
    ok = torch.equal(y.detach(), torch.cat(xs))                          # forward: rank-major concatenation
    (y * ws[rank]).sum().backward()
    want = sum(w[rank * B:(rank + 1) * B] for w in ws)                   # backward: every rank's gradient of MY rows, summed
    ok = ok and torch.allclose(x.grad, want, atol=1e-6)

    class M:  # DataParallel only attaches itself to the model and its towers
        pass
    m = M(); m.user_tower = M(); m.item_tower = M()
    dp = DataParallel(m)
    ok = ok and m.dp is dp and m.user_tower.dp is dp and dp.world == world and dp.rank == rank
    t = torch.full((3,), float(rank + 1), dtype=torch.float64)
    dp.reduce_sums(t)
    ok = ok and torch.equal(t, torch.full((3,), float(sum(range(1, world + 1))), dtype=torch.float64))
    rows, vals = dp.gather_sparse(torch.tensor([rank + 1, 0]), torch.full((2, 3), float(rank)))
    ok = ok and rows.tolist() == [1, 0, 2, 0] and vals[2].tolist() == [1.0, 1.0, 1.0]
    ok = ok and float(dp.global_loss(torch.tensor(0.5 * (rank + 1)))) == 1.5
    flat = torch.arange(10, dtype=torch.float32) * (rank + 1)              # only the listed runs are summed over replicas
    dp.reduce_dense_grad_(flat, [(0, 2), (7, 10)])
    want = torch.arange(10, dtype=torch.float32) * (rank + 1)
    want[0:2] = torch.arange(0, 2) * 3.0
    want[7:10] = torch.arange(7, 10) * 3.0
    ok = ok and torch.equal(flat, want)
    ok = ok and ShardedFlatIndex.exchange_width(100, 8) == 33 and ShardedFlatIndex.exchange_width(100, 1) == 100
    with open(os.path.join(tmp, f"dp{rank}"), "w") as fh:
        fh.write("1" if ok else "0")
    dist.destroy_process_group()


def test_data_parallel_plumbing_world_size_2_gloo(tmp_path):
    """The collectives of exact data-parallel training on CPU tensors (gloo): all-gathered rows with reduce-scattered
    gradients, summed statistics, gathered sparse rows, the global loss, the threshold-exchange width."""
    import torch.multiprocessing as mp
    port = 31500 + (os.getpid() % 2000)
    mp.spawn(_gloo_dp_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert [open(tmp_path / f"dp{r}").read() for r in range(2)] == ["1", "1"]


def test_feed_positives_csr_host_logic():
    """dict user -> positives (reference get_user_positive_items) -> CSR over users: duplicates collapse like the
    reference's set(), users without interactions get empty rows, out-of-range users are ignored."""
    import numpy as np
    from b200rec.feed import positives_csr
    indptr, items = positives_csr({0: [5, 3, 5, 1], 2: [7], 9: [1]}, n_users=4)
    assert indptr.tolist() == [0, 3, 3, 4, 4] and items.tolist() == [1, 3, 5, 7] and items.dtype == np.int32
    indptr, items = positives_csr({}, n_users=3)
    assert indptr.tolist() == [0, 0, 0, 0] and items.size >= 1      # never an empty device buffer


def test_feed_requires_cuda_and_big_enough_pools():
    import numpy as np
    import pytest
    from b200rec.feed import DeviceInteractionFeed
    with pytest.raises(RuntimeError, match="no CPU path"):
        DeviceInteractionFeed(np.zeros(4, np.int64), np.zeros(4, np.int64), np.ones(4), np.zeros((2, 3), np.float32),
                              np.zeros((5, 2), np.float32), {}, device="cpu")


def test_ixfi_file_format_round_trip(tmp_path):
    """Host side of the index persistence (SURVEY.md section 8 row f3): the `.faiss` file is faiss' IndexFlatIP layout
    ("IxFI", d, ntotal, two dummies, is_trained, metric 0, vector<float>), so faiss.read_index can open what we write
    and we can open what faiss.write_index wrote (reference retrieval.py:261,284)."""
    import struct
    from b200rec.retrieval import read_ixfi, write_ixfi
    rows = np.arange(35, dtype=np.float32).reshape(7, 5) / 3
    path = tmp_path / "x.faiss"
    write_ixfi(path, rows)
    raw = open(path, "rb").read()
    assert raw[:4] == b"IxFI" and len(raw) == 4 + 33 + 8 + rows.nbytes
    assert struct.unpack("<iqqqBi", raw[4:37]) == (5, 7, 1 << 20, 1 << 20, 1, 0)
    assert struct.unpack("<Q", raw[37:45]) == (35,)
    assert np.array_equal(read_ixfi(path), rows)
    open(path, "wb").write(b"IxF2" + raw[4:])
    with pytest.raises(ValueError, match="IxFI"):
        read_ixfi(path)
    open(path, "wb").write(raw[:-8])
    with pytest.raises(ValueError, match="truncated"):
        read_ixfi(path)
    bad_metric = raw[:33] + struct.pack("<i", 1) + raw[37:]
    open(path, "wb").write(bad_metric)
    with pytest.raises(ValueError, match="metric_type"):
        read_ixfi(path)


def test_flat_index_host_logic_without_a_gpu():
    """id mapping, the filter_ids post-pass and the engine bookkeeping with a stand-in for the device index."""
    from b200rec.retrieval import B200FlatIndex, RetrievalEngine

    class Fake:
        ntotal = 6

        def search(self, q, k, normalize=False):
            n = len(q)
            idx = np.tile(np.array([4, 2, 5, 0, 1, 3, -1, -1])[:k], (n, 1))
            return np.tile(np.linspace(1, 0, 8, dtype=np.float32)[:k], (n, 1)), idx

    eng = RetrievalEngine({"index_type": "b200", "embedding_dim": 4, "top_k": 3})
    ix = eng.index
    assert isinstance(ix, B200FlatIndex) and ix.dimension == 4
    ix.index, ix.current_size = Fake(), 6
    ix.id_map = {i: f"it{i}" for i in range(6)}
    ix.reverse_id_map = {v: k for k, v in ix.id_map.items()}
    q = np.zeros((2, 4), np.float32)
    ids, scores, m = eng.retrieve(q)
    assert ids == [["it4", "it2", "it5"]] * 2 and m["num_results"] == 6 and not m["cache_hit"]
    assert ix.search(q, k=8)[0][0] == ["it4", "it2", "it5", "it0", "it1", "it3"]          # -1 slots are dropped
    ids, scores = ix.search(q[0], k=2, filter_ids=["it5", "it1", "it3", "zzz"])           # post-filter over 2k = 4 rows
    assert ids == [["it5"]] and np.allclose(scores[0], [np.linspace(1, 0, 8)[2]])          # it1 / it3 lie beyond row 4
    ids, _ = ix.search(q[0], k=3, filter_ids=["it5", "it1", "it3", "it0"])                # 2k = 6 rows, first 3 survivors
    assert ids == [["it5", "it0", "it1"]]
    assert ix.search(q, k=1, filter_ids=["it3"])[0] == [[], []]                           # it3 is outside the 2 best rows
    del ix.id_map[2]
    ix._id_array = None
    assert ix.search(q, k=3)[0][0] == ["it4", "it5"]                                      # unmapped rows are skipped, not refilled
    assert eng.get_metrics()["total_queries"] == 1 and eng.get_metrics()["index_type"] == "b200"


class _OracleDeviceIndex:
    """CPU stand-in for b200rec.retrieval.FlatIPDeviceIndex in HOST-LOGIC tests only (tests may use the oracle; the
    product never does): same surface (`add(x, normalize)`, `search(q, k, normalize)`, `ntotal`, `reconstruct_n`)."""

    def __init__(self, d, storage="fp32", device=None, row_offset=0):
        from oracle.flat_ip import IndexFlatIP
        self.d, self._ix = d, IndexFlatIP(d)

    ntotal = property(lambda self: self._ix.ntotal)

    def add(self, x, normalize=False):
        from oracle.flat_ip import normalize_L2
        x = np.array(x, dtype=np.float32)
        self._ix.add(normalize_L2(x) if normalize else x)

    def search(self, q, k, normalize=False):
        from oracle.flat_ip import normalize_L2
        q = np.array(q, dtype=np.float32).reshape(-1, self.d)
        return self._ix.search(normalize_L2(q) if normalize else q, k)

    def reconstruct_n(self, i0=0, n=None):
        return self._ix.xb[i0:(None if n is None else i0 + n)].copy()


@pytest.mark.parametrize("metric", ["cosine", "ip"])
def test_drop_in_index_host_logic_matches_the_reference_wrapper_goldens(monkeypatch, tmp_path, metric):
    """The HOST side of B200FlatIndex / RetrievalEngine (casts, 1-D promotion, vectorised row -> id map, the filter_ids
    post-pass with k_search = min(2k, N), add, save / load through the IxFI file) against wrapper_small.npz — outputs of
    the REFERENCE's own FaissIndex / RetrievalEngine code — with the device index swapped for an oracle-backed stand-in,
    so this half of the drop-in boundary is pinned on CPU too (tests/test_gpu_index.py runs the real thing)."""
    import json
    from b200rec import retrieval
    monkeypatch.setattr(retrieval, "FlatIPDeviceIndex", _OracleDeviceIndex)
    g = np.load(os.path.join(ROOT, "tests", "golden", "wrapper_small.npz"))
    cases, allowed = json.loads(str(g["cases_json"])), json.loads(str(g["allowed_json"]))
    emb, extra, qry, N, D = g["emb"], g["extra"], g["qry"], int(g["N"]), int(g["D"])

    def same(got, want):
        assert got[0] == want[0], "item ids differ"
        for a, b in zip(got[1], want[1]):
            assert len(a) == len(b) and np.allclose(a, b, rtol=1e-6, atol=2e-6)

    ix = retrieval.B200FlatIndex({"dimension": D, "index_factory": "IVF1024,Flat", "metric": metric})
    with pytest.raises(ValueError, match="Index not built yet"):
        ix.search(qry, k=3)
    with pytest.raises(ValueError, match="No index to save"):
        ix.save(str(tmp_path / "never"))
    ix.build(emb.copy(), [f"item_{i}" for i in range(N)])
    same(ix.search(qry.copy(), k=10), cases[f"{metric}_k10"])
    same(ix.search(qry[0].copy(), k=5), cases[f"{metric}_1d_k5"])
    same(ix.search(qry.astype(np.float64), k=7, filter_ids=allowed), cases[f"{metric}_filter_k7"])
    assert ix.search(qry[:2].copy(), k=4, filter_ids=[]) == ([[], []], [[], []])
    ix.save(str(tmp_path / "idx"))                       # IxFI + pkl round trip keeps rows, ids and answers
    ix2 = retrieval.B200FlatIndex({"dimension": D, "metric": metric})
    ix2.load(str(tmp_path / "idx"))
    assert ix2.current_size == N and ix2.id_map[3] == "item_3"
    same(ix2.search(qry.copy(), k=10), cases[f"{metric}_k10"])
    ix.add(extra.copy(), [f"new_{i}" for i in range(len(extra))])
    same(ix.search(qry.copy(), k=10), cases[f"{metric}_after_add_k10"])
    assert ix.current_size == cases[f"{metric}_size"]
    if metric == "cosine":
        eng = retrieval.RetrievalEngine({"index_type": "faiss", "embedding_dim": D,
                                         "faiss": {"index_factory": "Flat", "metric": "cosine"}})
        eng.build_index(emb.copy(), [f"item_{i}" for i in range(N)])
        ids, scores, metrics = eng.retrieve(qry[:2].copy(), k=6)
        same((ids, scores), cases["engine_retrieve_k6"])
        assert sorted(metrics.keys()) == cases["engine_metrics_keys"] and metrics["num_results"] == 12


def test_bench_host_logic_without_a_gpu():
    """bench.py pieces that need no GPU: both arms print the same `config`, a failing extra block is recorded inside the
    single-GPU line but stays fatal under torchrun, the peaks loader never raises, the CPU arm picks the C reservoir."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    assert bench.primary_config(8)["workload"].endswith("over 8 GPU(s)") and bench.primary_config(1)["seed"] == bench.SEED
    extra = {}

    def boom(x):
        raise RuntimeError("no memory for " + x)

    bench.run_block(extra, 1, "ok", lambda v: {"value": v}, 3)
    bench.run_block(extra, 1, "bad", boom, "cfg4")
    assert extra["ok"] == {"value": 3} and "no memory for cfg4" in extra["bad"]["error"]
    with pytest.raises(RuntimeError):
        bench.run_block(extra, 2, "bad2", boom, "serve")
    peaks = bench._peaks()
    assert peaks["tflops"] > 0 and peaks["hbm_gbs"] > 0 and peaks["tflops_burst"] >= peaks["tflops"]
    search, what = bench._cpu_search()
    assert search.__name__ == "search_reservoir" and "flat_select.c" in what
    qps, dt, what2 = bench.cpu_retrieval_baseline(1 << 17, 64, 2)          # the GPU arm's cpu_baseline leg, tiny sample
    assert qps > 0 and dt > 0 and what2 == what
