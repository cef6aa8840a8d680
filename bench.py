#!/usr/bin/env python
"""bench.py — headline benchmark of the B200 two-tower hot path (contract: ONE JSON line on rank 0).

Primary workload (BASELINE.json config 3): exact inner-product top-100 over a 10 M x 128 bf16 catalogue, query batch
4096, catalogue row-sharded over the N GPUs of one box (total work fixed => "strong" scaling).
  value  = whole-job QPS with the query operand resident in HBM (CUDA events, max over ranks)
  e2e    = the same through the faiss-shaped plugin call with HOST numpy buffers (`index.search_stream`: numpy queries
           in, (D, I) numpy out; every batch's host->device and device->host copies are inside the timed region,
           double-buffered against the neighbouring batches' searches); `e2e_sync_call` = one blocking
           `index.search(q, k)` per step
  parity_checked = 32 of the timed 4096 queries re-searched on the host (oracle sgemm + exact select over every shard)
Extra blocks in the same line (each with its own `roofline` and, at N = 1, `cpu_baseline`):
  train       config 2  synthetic 1 M users x 100 K items, dim 64, batch 8192 per GPU, in-batch negatives (DP at N > 1)
  train_ml1m  config 1  MovieLens-1M-shaped step through the device feed;  epoch_ml1m: a full epoch + exact top-100 eval
  train_cfg4  config 4  50 M / 5 M-row tables, dim 128, batch 8192 per GPU, row-sparse tables (DP at N > 1)
  serve       config 5  user-tower forward + 100 M x 64 sharded top-1000, Q sweep
`--impl reference` times the reference's CPU path on the host cores: flat search = faiss-cpu's blocked sgemm + k-select
restated (oracle/flat_ip.search_reservoir; faiss itself is not installable offline), training = the imported reference
model + its trainer's step body on torch-CPU (baseline/_ref, staged by __graft_entry__.build()).

  python bench.py --gpus 1 --steps 20 --warmup 5
  python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 bench.py --gpus 8
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_ITEMS = 10_000_000
DIM = 128
N_QUERIES = 4096
TOPK = 100
SEED = 1234
METRIC = "top-100 exact-IP QPS over 10M items"


def primary_config(world: int) -> dict:
    """`config` of the primary line: the same dict on both arms (the CPU arm times a bounded sample OF this workload and
    says which in `cpu_baseline.sample`)."""
    return {"workload": "exact IP top-100 retrieval, 10M items x 128-dim bf16, query batch 4096, "
                        f"catalogue row-sharded over {world} GPU(s)",
            "l2": "catalogue shard (>= 320 MB) exceeds L2 between iterations", "seed": SEED}


def _peaks():
    """Roofline denominators: the driver-measured copy bandwidth and bf16 throughput of this pool's B200s
    (MEASURED_PEAKS.json), else the fallback B200_PROFILING.md states.  Never raises: the line being printed with the
    fallback peaks beats losing a finished measurement to a malformed file."""
    fallback = {"hbm_gbs": 6650.0, "tflops": 1400.0, "tflops_burst": 1650.0, "source": "fallback (B200_PROFILING.md)"}
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            p = json.load(fh)
        burst = float(p["bf16_tflops"])
        return {"hbm_gbs": float(p["hbm_gbs"]), "tflops": float(p.get("bf16_tflops_sustained") or burst),
                "tflops_burst": burst, "source": "measured (MEASURED_PEAKS.json: sustained bf16, copy bandwidth)"}
    except Exception:  # noqa: BLE001 - absent, unreadable or partial file
        return fallback


def host_threads() -> int:
    """All host cores, set explicitly: torchrun exports OMP_NUM_THREADS=1, which would silently throttle the CPU arm."""
    n = os.cpu_count() or 1
    torch.set_num_threads(n)
    return n


class ClockSampler:
    """nvidia-smi clocks / power / throttle reasons sampled DURING the timed region."""

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index
        self.thread = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return

        def pump():
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])

        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, pw, smax, reasons = [], [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                smax = float(r[1])
                pw.append(float(r[2]))
                for name, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_median": float(np.median(pw)) if pw else None,
                "power_w_max": float(np.max(pw)) if pw else None}


# ------------------------------------------------------------------------------------------------ data
def make_queries_host(n: int = N_QUERIES, dim: int = DIM, seed: int = SEED) -> torch.Tensor:
    g = torch.Generator().manual_seed(seed)
    return torch.nn.functional.normalize(torch.randn(n, dim, generator=g), dim=1)


def make_catalogue_shard(lo: int, hi: int, device, n_total: int = N_ITEMS, dim: int = DIM, seed: int = SEED) -> torch.Tensor:
    """Rows [lo, hi) of the synthetic catalogue normalize(N(0,1)) -> bf16; generated block-wise from (seed, block) so
    any sharding sees the same global rows."""
    out = torch.empty((hi - lo, dim), dtype=torch.bfloat16, device=device)
    blk = 1 << 20
    b0 = lo // blk
    while b0 * blk < hi:
        s, e = b0 * blk, min((b0 + 1) * blk, n_total)
        g = torch.Generator(device=device).manual_seed(seed * 1000003 + b0)
        x = torch.nn.functional.normalize(torch.randn(e - s, dim, device=device, generator=g), dim=1).to(torch.bfloat16)
        a, b = max(s, lo), min(e, hi)
        out[a - lo:b - lo] = x[a - s:b - s]
        b0 += 1
    return out


def zipf_ids(rng, n, hi):
    return np.clip(rng.zipf(1.05, size=n), 1, hi).astype(np.int64)


# ------------------------------------------------------------------------------------------------ CPU baselines
def cpu_retrieval_baseline(rows: int, queries: int, threads: int):
    """Flat IP top-100 the way faiss-cpu lays it out (blocked sgemm + k-select per block, all host cores) on a bounded
    sample; QPS scaled linearly to 10 M rows (the work per query is proportional to the catalogue)."""
    search, what = _cpu_search()
    cat, qry = _cpu_sample(rows, queries)
    search(cat[: 1 << 17], qry[:64], TOPK, threads)   # warm the thread pools
    search(cat, qry, TOPK, threads)
    reps = 3
    t0 = time.perf_counter()
    for _ in range(reps):
        search(cat, qry, TOPK, threads)
    dt = (time.perf_counter() - t0) / reps
    return queries / (dt * (N_ITEMS / rows)), dt, what


def _reference_modules():
    """The UNMODIFIED reference model / trainer modules staged under baseline/_ref (None when not staged)."""
    ref = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isfile(os.path.join(ref, "src", "models", "two_tower.py")):
        return None
    if ref not in sys.path:
        sys.path.insert(0, ref)
    import importlib
    return {"two_tower": importlib.import_module("src.models.two_tower"),
            "utils": importlib.import_module("src.training.utils"),
            "trainer": importlib.import_module("src.training.trainers.two_tower")}


def cpu_train_baseline_cfg2(threads: int, steps: int = 3):
    """Config 2 on the host cores: the IMPORTED reference model (1 M / 100 K-row embedding tables at the reference's own
    row width heuristic min(50, .)) and the step body of its TwoTowerTrainer.train_epoch (trainers/two_tower.py:98-151:
    towers, in-batch loss, zero_grad, backward, clip_grad_norm_(1.0), Adam(lr 1e-3, wd 1e-5).step) on torch-CPU.  The
    reference trainer itself feeds no categorical ids, so its step body is driven here with the config-2 id tensors."""
    mods = _reference_modules()
    B, NU, NI, FD = 8192, 1_000_000, 100_000, 16
    rng = np.random.default_rng(SEED)
    if mods is None:
        return None
    tt = mods["two_tower"]
    torch.manual_seed(SEED)
    ut = tt.UserTower(FD, 64, [128, 64], 0.2, "relu", {"user_id": NU})
    it = tt.ItemTower(FD, 64, [128, 64], 0.2, "relu", {"item_id": NI}, use_content_embedding=False)
    model = tt.TwoTowerModel(ut, it, temperature=0.05)
    opt = torch.optim.Adam(model.parameters(), lr=1e-3, weight_decay=1e-5)
    model.train()
    uf, pf = torch.randn(B, FD), torch.randn(B, FD)
    uid, iid = torch.from_numpy(zipf_ids(rng, B, NU)), torch.from_numpy(zipf_ids(rng, B, NI))

    def step():
        u = model.get_user_embeddings({"numerical": uf, "categorical": {"user_id": uid}})
        p = model.get_item_embeddings({"numerical": pf, "categorical": {"item_id": iid}})
        loss = model.in_batch_negative_loss(u, p)
        opt.zero_grad()
        loss.backward()
        torch.nn.utils.clip_grad_norm_(model.parameters(), max_norm=1.0)
        opt.step()
        return float(loss.item())

    step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    return {"value": B / dt, "unit": "samples/s", "cores": threads, "kind": "reference",
            "sample": f"{steps} steps of the imported reference TwoTowerModel (baseline/_ref) + its trainer's step body "
                      f"(in-batch loss, clip, dense Adam) on torch-CPU at batch {B}, tables 1M / 100K rows",
            "ms_per_step": dt * 1e3}


def cpu_train_baseline_ml1m(threads: int, steps: int = 3):
    """Config 1 step on the host cores: the imported reference TwoTowerTrainer.train_epoch over pre-built batches
    (batch 1024 x 16 negatives, 0.7 explicit + 0.3 in-batch), i.e. the reference's model time WITHOUT its Python feed."""
    mods = _reference_modules()
    if mods is None:
        return None
    torch.manual_seed(SEED)
    model = mods["utils"].create_two_tower_model_for_training(3, 20, {"embedding_dim": 128, "hidden_layers": [256, 128],
                                                                      "dropout_rate": 0.2, "temperature": 0.05})
    batches = [{"user_features": torch.randn(1024, 3), "pos_item_features": torch.randn(1024, 20),
                "neg_item_features": torch.randn(1024, 16, 20)} for _ in range(steps)]
    tr = mods["trainer"].TwoTowerTrainer(model, batches, [], {"learning_rate": 1e-3, "weight_decay": 1e-5,
                                                              "checkpoint_dir": "/tmp/b200rec_ref_ckpt"}, device="cpu")
    tr.train_loader = batches[:1]
    tr.train_epoch(0)
    tr.train_loader = batches
    t0 = time.perf_counter()
    tr.train_epoch(1)
    dt = (time.perf_counter() - t0) / steps
    return {"value": 1024 / dt, "unit": "samples/s", "cores": threads, "kind": "reference",
            "sample": f"{steps} batches through the imported reference TwoTowerTrainer.train_epoch on torch-CPU "
                      "(batch 1024 x 16 negatives, mixed loss), batches pre-built: model time without the reference's feed",
            "ms_per_step": dt * 1e3}


def _cpu_search():
    """(function, description) of the CPU flat search both CPU legs time: faiss-cpu's layout restated — blocked MKL sgemm
    + the C reservoir result handler (oracle/csrc/flat_select.c); torch.topk per block if no C compiler is around."""
    from oracle import flat_ip
    try:
        flat_ip._select_lib()
        return flat_ip.search_reservoir, ("oracle/flat_ip.search_reservoir = faiss-cpu's IndexFlatIP layout restated (blocked MKL "
                                          "sgemm + C reservoir k-select, oracle/csrc/flat_select.c; faiss-cpu is not "
                                          "installable offline)")
    except Exception:  # noqa: BLE001 - no gcc on this host: the slower torch.topk select
        return flat_ip.search_blocked, ("oracle/flat_ip.search_blocked = faiss-cpu's IndexFlatIP layout restated (blocked MKL "
                                        "sgemm + torch.topk per block; the C reservoir select could not be built here; "
                                        "faiss-cpu is not installable offline)")


def _cpu_sample(rows: int, queries: int):
    g = torch.Generator().manual_seed(SEED)
    cat = torch.nn.functional.normalize(torch.randn(rows, DIM, generator=g), dim=1)
    qry = torch.nn.functional.normalize(torch.randn(queries, DIM, generator=g), dim=1)
    return cat, qry


def run_reference(args, rank: int, world: int):
    """CPU arm: W warm-up + EXACTLY K timed steps, each step one flat search of a bounded sample of config 3 (the whole
    4096-query batch against 1 M of the 10 M rows, fp32, all host threads); QPS scaled linearly in the rows.  The
    sample shrinks (never the step count) if K steps of it would not end within a few minutes on this host."""
    if rank != 0:
        return
    search, what = _cpu_search()
    threads = host_threads()
    rows, queries = 1_000_000, N_QUERIES
    steps, warmup = args.steps, max(args.warmup, 0)
    cat, qry = _cpu_sample(rows, queries)
    search(cat[: 1 << 17], qry[:64], TOPK, threads)   # start the thread pools
    t0 = time.perf_counter()
    search(cat, qry, TOPK, threads)
    probe = time.perf_counter() - t0
    budget_s = 150.0
    if probe * (steps + warmup) > budget_s:
        rows = max(1 << 17, int(rows * budget_s / (probe * (steps + warmup))) // (1 << 17) * (1 << 17))
        cat = cat[:rows].contiguous()
    for _ in range(warmup):
        search(cat, qry, TOPK, threads)
    t_all = time.perf_counter()
    for _ in range(steps):
        search(cat, qry, TOPK, threads)
    dt = (time.perf_counter() - t_all) / steps
    ms = dt * 1e3
    v = float(queries / (dt * (N_ITEMS / rows)))
    sample = (f"{queries} queries x {rows} rows fp32 per step on {threads} threads (OMP/MKL threads set explicitly), "
              f"{what}, QPS scaled linearly to {N_ITEMS} rows")
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "queries/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": primary_config(world),
            "cpu_baseline": {"value": v, "unit": "queries/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if not args.no_train:
        try:
            line["train"] = cpu_train_baseline_cfg2(threads)
            line["train_ml1m"] = cpu_train_baseline_ml1m(threads)
        except Exception as exc:  # noqa: BLE001 - the retrieval line must still be printed
            line["train_error"] = repr(exc)[:300]
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ helpers
class Ctx:
    def __init__(self, device, world, rank):
        self.device, self.world, self.rank = device, world, rank

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, *vals):
        t = torch.tensor(list(vals), dtype=torch.float64, device=self.device)
        if self.world > 1:
            import torch.distributed as dist
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t.tolist()]


def timed(ctx: Ctx, fn, steps: int, warmup: int) -> float:
    """ms per step of fn(i): barrier + synchronize on both sides, CUDA events, max over ranks."""
    for i in range(warmup):
        fn(i)
    ctx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        fn(i)
    e1.record()
    ctx.barrier()
    return ctx.max_over_ranks(e0.elapsed_time(e1) / steps)[0]


# ------------------------------------------------------------------------------------------------ parity of the timed run
def parity_check(ctx: Ctx, index, q_host: torch.Tensor, scores: torch.Tensor, ids: torch.Tensor, n_check: int = 32):
    """Re-search `n_check` of the timed queries on the HOST: every rank scores its own catalogue shard with the oracle
    (numpy sgemm + exact select on the bf16-rounded rows upcast to fp32), the per-shard lists are merged on rank 0 and
    compared with what the GPU path returned for those queries (ids exact except inside score ties within 1e-5)."""
    import torch.distributed as dist
    from oracle.flat_ip import IndexFlatIP, merge_topk
    g = torch.Generator().manual_seed(SEED + 17)
    pick = torch.randperm(q_host.shape[0], generator=g)[:n_check].sort().values
    qs = q_host[pick].to(torch.bfloat16).to(torch.float32).numpy()
    run_s = np.full((n_check, TOPK), -np.finfo(np.float32).max, np.float32)
    run_i = np.full((n_check, TOPK), -1, np.int64)
    t0 = time.perf_counter()
    chunk = 1 << 20
    for r0 in range(0, index.ntotal, chunk):
        rows = index._cat[r0:min(index.ntotal, r0 + chunk), : index.d].float().cpu().numpy()
        ix = IndexFlatIP(index.d, db_block=1 << 17)
        ix.add(rows)
        s, i = ix.search(qs, TOPK)
        i = np.where(i >= 0, i + r0 + index.row_offset, -1)
        run_s, run_i = merge_topk([run_s, s], [run_i, i], TOPK)
    if ctx.world > 1:
        ts, ti = torch.from_numpy(run_s).to(ctx.device), torch.from_numpy(run_i).to(ctx.device)
        gs = [torch.empty_like(ts) for _ in range(ctx.world)]
        gi = [torch.empty_like(ti) for _ in range(ctx.world)]
        dist.all_gather(gs, ts)
        dist.all_gather(gi, ti)
        run_s, run_i = merge_topk([x.cpu().numpy() for x in gs], [x.cpu().numpy() for x in gi], TOPK)
    got_s, got_i = scores[pick.to(scores.device)].cpu().numpy(), ids[pick.to(ids.device)].cpu().numpy()
    diff = got_i != run_i
    ties_ok = bool((np.abs(got_s - run_s)[diff] <= 1e-5).all())
    ok = bool(np.allclose(got_s, run_s, atol=2e-5, rtol=0) and ties_ok and diff.mean() <= 0.01)
    return {"queries": int(n_check), "ok": ok, "ids_differing_inside_ties": int(diff.sum()),
            "max_abs_score_diff": float(np.abs(got_s - run_s).max()), "seconds": round(time.perf_counter() - t0, 2),
            "checker": "oracle/flat_ip.IndexFlatIP over every shard (host), merged on rank 0"}


# ------------------------------------------------------------------------------------------------ training blocks
def _train_roofline(ms: float, flops: float, bytes_: float, note: str):
    pk = _peaks()
    t_tensor = flops / (pk["tflops"] * 1e12) * 1e3
    t_hbm = bytes_ / (pk["hbm_gbs"] * 1e9) * 1e3
    bound = "hbm" if t_hbm >= t_tensor else "tensor"
    if bound == "hbm":
        achieved, peak, unit = bytes_ / (ms * 1e-3) / 1e9, pk["hbm_gbs"], "GB/s"
    else:
        achieved, peak, unit = flops / (ms * 1e-3) / 1e12, pk["tflops"], "TFLOP/s"
    return {"bound": bound, "achieved": achieved, "peak": peak, "unit": unit, "frac": achieved / peak, "traffic": None,
            "scope": "whole training step (launch-bound chains of small kernels: no single kernel dominates)",
            "algorithmic_flops": flops, "algorithmic_bytes": bytes_, "tensor_floor_ms": t_tensor, "hbm_floor_ms": t_hbm,
            "frac_of_tensor_peak": flops / (ms * 1e-3) / 1e12 / pk["tflops"],
            "frac_of_hbm_peak": bytes_ / (ms * 1e-3) / 1e9 / pk["hbm_gbs"], "note": note, "peak_source": pk["source"]}


def _make_cfg_model(device, FD, NU, NI, edim, hidden, E, sparse_tables):
    from b200rec.training_utils import create_two_tower_model_for_training
    cfg = {"embedding_dim": E, "hidden_layers": hidden, "dropout_rate": 0.2, "temperature": 0.05,
           "user_categorical_features": {"user_id": NU}, "item_categorical_features": {"item_id": NI},
           "embedding_dims": {"user_id": edim, "item_id": edim}, "sparse_tables": sparse_tables}
    torch.manual_seed(SEED)
    with torch.device(device):          # parameters are created and initialised on the GPU (a 50 M-row table never
        model = create_two_tower_model_for_training(FD, FD, cfg)   # visits the host)
    return model


def run_table_train_block(ctx: Ctx, steps: int, warmup: int, cpu_baseline: bool, *, name: str, NU: int, NI: int,
                          edim: int, hidden, E: int, sparse_tables: bool, check_dp: bool):
    """One data-parallel training configuration with id-embedding tables (configs 2 and 4): batch 8192 PER GPU,
    in-batch negatives over the GLOBAL batch, exact data parallel at N > 1 (b200rec.dist.DataParallel)."""
    import torch.distributed as dist
    from b200rec import _native as N
    from b200rec.trainer import TwoTowerTrainer
    device, world, rank = ctx.device, ctx.world, ctx.rank
    B, FD = 8192, 16
    model = _make_cfg_model(device, FD, NU, NI, edim, hidden, E, sparse_tables)
    trainer = TwoTowerTrainer(model, [], [], {"learning_rate": 1e-3, "weight_decay": 1e-5,
                                              "checkpoint_dir": "/tmp/b200rec_bench_ckpt"}, device=str(device))
    if world > 1:
        from b200rec.dist import DataParallel
        DataParallel(model)
    model.train()
    rng = np.random.default_rng(SEED + 1000 * rank)
    torch.manual_seed(SEED + 1000 * rank)   # features differ per replica; parameters were initialised identically above
    pool = 8
    host = [{"uf": torch.randn(B, FD).pin_memory(), "pf": torch.randn(B, FD).pin_memory(),
             "uid": torch.from_numpy(zipf_ids(rng, B, NU)).pin_memory(),
             "iid": torch.from_numpy(zipf_ids(rng, B, NI)).pin_memory()} for _ in range(pool)]
    dev = [{k: v.to(device) for k, v in b.items()} for b in host]

    def step_dev(b):
        return trainer.train_step(b["uf"], b["pf"], None, {"user_id": b["uid"]}, {"item_id": b["iid"]})

    dp_check = None
    if world > 1 and check_dp:
        # step 1 runs without dropout (masks are per replica by design) so that it can be replayed by one process
        for t in (model.user_tower, model.item_tower):
            t.dropout_rate = 0.0
        first_loss = step_dev(dev[0])
        dp_check = _dp_first_step_check(ctx, first_loss, dev[0], FD, NU, NI, edim, hidden, E, sparse_tables)
        for t in (model.user_tower, model.item_tower):
            t.dropout_rate = 0.2
    else:
        step_dev(dev[0])
    torch.cuda.synchronize()
    lc0 = N.launch_count()
    step_dev(dev[1])
    kernels_per_step = N.launch_count() - lc0      # library kernels of one eager step (a graph replays the same nodes)
    graph = trainer.enable_cuda_graph(warm_steps=1)
    ms = timed(ctx, lambda i: step_dev(dev[i % pool]), steps, max(warmup, 3))
    # end to end: host batches (pinned) -> device every step, loss read back every step
    ctx.barrier()
    t0 = time.perf_counter()
    for i in range(steps):
        b = {k: v.to(device, non_blocking=True) for k, v in host[i % pool].items()}
        float(step_dev(b).item())
    ctx.barrier()
    e2e_ms = ctx.max_over_ranks((time.perf_counter() - t0) / steps * 1e3)[0]
    # algorithmic work of ONE replica's step (SURVEY.md section 8d): towers 6 * sum(in*out) FLOP per sample and pass,
    # in-batch loss 6 * B_local * B_global * E; bytes = optimiser traffic (24-28 B per densely updated parameter; row-sparse
    # tables touch 28 B per element of a touched row) + embedding gather / scatter + activations
    dims = [FD + edim] + list(hidden) + [E]
    macs = sum(a * b for a, b in zip(dims[:-1], dims[1:]))
    flops = 2 * 6 * B * macs + 6.0 * B * (B * world) * E
    mlp_params = 2 * sum(a * b + b for a, b in zip(dims[:-1], dims[1:]))
    table_params = (NU + 1 + NI + 1) * edim
    # dense tables: p, m, v read + written = 24 B per parameter (the gradient is read, and reset, on touched rows only:
    # b200rec_adam_table); MLP parameters 28 B (g read as well)
    dense_bytes = 28.0 * mlp_params + (0.0 if sparse_tables else 24.0 * table_params + 2 * 8.0 * B * edim * world)
    sparse_bytes = (28.0 * 2 * B * edim * world) if sparse_tables else 0.0
    act_bytes = 4.0 * B * sum(dims) * 2 * 3
    bytes_ = dense_bytes + sparse_bytes + act_bytes + 2 * B * (8 + 2 * 4 * edim)
    h2d = sum(v.numel() * v.element_size() for v in host[0].values())
    out = {"metric": "train samples/s", "value": world * B / ms * 1e3, "unit": "samples/s", "ms_per_step": ms,
           "n_gpus": world, "scaling": "weak",
           "config": {"workload": f"{name}: {NU} users x {NI} items, id-embedding dim {edim}, E {E}, hidden {list(hidden)}, "
                                  f"batch {B} per GPU (global {world * B}), in-batch negatives over the global batch, "
                                  "fp32-grade split-bf16 GEMMs, " +
                                  ("row-sparse Adam on the touched table rows (dense Adam on the MLP)" if sparse_tables
                                   else "dense Adam + clip over ALL parameters (reference semantics)") +
                                  (", exact data parallel: synced BatchNorm statistics, all-gathered negatives, summed "
                                   "gradients" if world > 1 else "")},
           "e2e": {"value": world * B / e2e_ms * 1e3, "unit": "samples/s", "h2d_bytes_per_step": h2d * world,
                   "d2h_bytes_per_step": 4 * world},
           "gpu_launches_per_step": int(kernels_per_step), "cuda_graph": bool(graph),
           "dtype": "f32 (bf16x6 split products, fp32 accumulate)",
           "roofline": _train_roofline(ms, flops, bytes_, "per replica; bytes dominated by " +
                                       ("the touched rows' Adam state" if sparse_tables else "dense Adam over both tables"))}
    if dp_check is not None:
        out["dp_check"] = dp_check
    if cpu_baseline:
        try:
            out["cpu_baseline"] = cpu_train_baseline_cfg2(host_threads())
        except Exception as exc:  # noqa: BLE001
            out["cpu_baseline"] = {"error": repr(exc)[:200]}
    trainer.release_graphs()
    del trainer, model, dev
    torch.cuda.empty_cache()
    return out


def _dp_first_step_check(ctx: Ctx, dp_loss, batch, FD, NU, NI, edim, hidden, E, sparse_tables):
    """The data-parallel loss of step 1 is (a) identical on every rank and (b) what ONE process computes on the
    concatenated global batch: rank 0 replays the forward of step 1 without data parallelism on an identically
    initialised model (same seed) and compares."""
    import torch.distributed as dist
    world, rank, device = ctx.world, ctx.rank, ctx.device
    losses = [torch.empty_like(dp_loss.reshape(1)) for _ in range(world)]
    dist.all_gather(losses, dp_loss.detach().reshape(1))
    same = all(torch.equal(losses[0], x) for x in losses)
    gathered = {}
    for k in ("uf", "pf", "uid", "iid"):
        parts = [torch.empty_like(batch[k]) for _ in range(world)]
        dist.all_gather(parts, batch[k])
        gathered[k] = torch.cat(parts)
    rel = None
    if rank == 0:
        ref = _make_cfg_model(device, FD, NU, NI, edim, hidden, E, sparse_tables).to(device)
        ref.train()
        for t in (ref.user_tower, ref.item_tower):
            t.dropout_rate = 0.0
        with torch.no_grad():
            u = ref.get_user_embeddings({"numerical": gathered["uf"], "categorical": {"user_id": gathered["uid"]}})
            p = ref.get_item_embeddings({"numerical": gathered["pf"], "categorical": {"item_id": gathered["iid"]}})
            single = ref.in_batch_negative_loss(u, p)
        rel = abs(float(single.item()) - float(dp_loss.item())) / abs(float(single.item()))
        del ref
    torch.cuda.empty_cache()
    return {"loss_identical_on_all_ranks": bool(same), "rel_diff_vs_single_process_forward": rel,
            "ok": bool(same and (rel is None or rel <= 1e-6)),
            "note": "step 1 (dropout off: masks are per replica by design) replayed by ONE process on rank 0 over the "
                    "all-gathered global batch with an identically initialised model (training-mode BatchNorm)"}


def run_ml1m_block(ctx: Ctx, steps: int, warmup: int, cpu_baseline: bool):
    """BASELINE config 1 shape (MovieLens-1M: 6,040 users x 3 features, 3,416 movies x 20 features, 799,688 training
    interactions, batch 1024, 16 sampled negatives, E=128, hidden [256,128], loss 0.7 explicit + 0.3 in-batch) on a
    synthetic interaction table, fed by the device-side feed (b200rec.feed: negative sampling + feature gathers on the
    GPU) — the step the reference runs at ~0.19 s of model time + 0.46 s of Python sampling per batch and worker."""
    from b200rec.feed import DeviceInteractionFeed
    from b200rec.trainer import TwoTowerTrainer
    from b200rec.training_utils import create_two_tower_model_for_training
    device = ctx.device
    NU, NM, NI, B, R = 6040, 3416, 799_688, 1024, 16
    rng = np.random.default_rng(SEED)
    u = rng.integers(0, NU, NI)
    m = np.minimum(rng.zipf(1.2, NI) - 1, NM - 1)
    lab = np.ones(NI, dtype=np.float64)
    uf = rng.standard_normal((NU, 3)).astype(np.float32)
    mf = rng.standard_normal((NM, 20)).astype(np.float32)
    pos = {}
    for a, b in zip(u.tolist(), m.tolist()):
        pos.setdefault(a, []).append(b)
    torch.manual_seed(SEED)
    model = create_two_tower_model_for_training(3, 20, {"embedding_dim": 128, "hidden_layers": [256, 128],
                                                          "dropout_rate": 0.2, "temperature": 0.05})
    feed = DeviceInteractionFeed(u, m, lab, uf, mf, pos, num_items=NM, num_negatives=R, batch_size=B, seed=SEED,
                                 device=str(device))
    trainer = TwoTowerTrainer(model, feed, [], {"learning_rate": 1e-3, "weight_decay": 1e-5,
                                                "checkpoint_dir": "/tmp/b200rec_bench_ckpt"}, device=str(device))
    model.train()
    trainer.enable_cuda_graph(warm_steps=2)
    it = iter(feed)
    for _ in range(max(warmup, 3)):
        b = next(it)
        trainer.train_step(b["user_features"], b["pos_item_features"], b["neg_item_features"])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        b = next(it)
        loss = trainer.train_step(b["user_features"], b["pos_item_features"], b["neg_item_features"])
    float(loss.item())
    dt = (time.perf_counter() - t0) / steps
    feed.check()
    macs_u = 3 * 256 + 256 * 128 + 128 * 128
    macs_i = 20 * 256 + 256 * 128 + 128 * 128
    flops = 6.0 * (B * macs_u + (B + B * R) * macs_i) + 6.0 * B * B * 128 + 6.0 * B * (R + 1) * 128
    params = sum(p.numel() for p in model.parameters())
    bytes_ = 28.0 * params + 4.0 * (B * (3 + 256 + 128 + 128) + (B + B * R) * (20 + 256 + 128 + 128)) * 2 * 3
    out = {"metric": "train samples/s", "value": B / dt, "unit": "samples/s", "ms_per_step": dt * 1e3,
           "epoch_s_at_this_rate": NI / B * dt,
           "config": {"workload": "MovieLens-1M shape (synthetic interactions): batch 1024 x 16 sampled negatives, E=128, "
                                  "hidden [256,128], 0.7 explicit + 0.3 in-batch loss; batches built on the GPU by "
                                  "b200rec.feed (negative sampling + feature gathers), step replayed as one CUDA graph, wall clock "
                                  "including the feed"},
           "roofline": _train_roofline(dt * 1e3, flops, bytes_, "5.97 GFLOP / 28 MB per step: microseconds of work, the "
                                                                   "step is bound by launch latency of its kernel chain")}
    if cpu_baseline:
        from oracle.feed import make_batch
        np.random.seed(SEED)
        t0 = time.perf_counter()
        make_batch(list(range(512)), u, m, lab, uf, mf, pos, NM, R, True)
        per_sample = (time.perf_counter() - t0) / 512
        out["cpu_baseline_feed"] = {"value": 1.0 / per_sample, "unit": "samples/s", "cores": 1, "kind": "port",
                                    "sample": "512 samples of oracle/feed.py (sample_negative_items + __getitem__ + "
                                              "collate_fn restated): the reference's FEED alone, one DataLoader worker"}
        try:
            out["cpu_baseline"] = cpu_train_baseline_ml1m(host_threads())
        except Exception as exc:  # noqa: BLE001
            out["cpu_baseline"] = {"error": repr(exc)[:200]}
    del trainer, model, feed
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------------ config 1: epoch + eval
def synth_ratings(path: str, users_dat: str, movies_dat: str, n: int = 1_000_209, seed: int = SEED) -> None:
    """ratings.dat is not shipped with the reference (.MISSING_LARGE_BLOBS): synthesise `UserID::MovieID::Rating::
    Timestamp` rows over the real user / movie ids (SURVEY.md section 8c), fixed seed.  The towers of the ML-1M
    configuration see FEATURES only (gender / age / occupation, genres / year), so the synthetic preferences are a
    fixed random bilinear form of exactly those fields: affinity(u, m) = [gender, age, occupation one-hot](u) . W .
    genres(m).  Each user draws a log-normal number (>= 20, as in ML-1M) of distinct movies with probability
    proportional to popularity x exp(1.5 affinity) (Gumbel top-k) and rates them 1-5 around 3.1 + 0.9 affinity;
    timestamps 2000-04-25 .. 2003-02-28.  A model can therefore learn something, and its scores do not collapse into
    ties (with preference-free random ratings every user's top-100 was decided by 1e-8 score differences)."""
    rng = np.random.default_rng(seed)
    urows = [l.strip().split("::") for l in open(users_dat, encoding="latin-1") if l.strip()]
    mrows = [l.strip().split("::") for l in open(movies_dat, encoding="latin-1") if l.strip()]
    uids = np.array([int(r[0]) for r in urows])
    mids = np.array([int(r[0]) for r in mrows])
    genres = sorted({g for r in mrows for g in r[2].split("|")})
    gmat = np.zeros((len(mrows), len(genres)), dtype=np.float32)
    for i, r in enumerate(mrows):
        for g in r[2].split("|"):
            gmat[i, genres.index(g)] = 1.0
    gmat /= np.sqrt(gmat.sum(1, keepdims=True))
    ufe = np.zeros((len(urows), 2 + 21), dtype=np.float32)
    for i, r in enumerate(urows):
        ufe[i, 0] = 1.0 if r[1] == "M" else -1.0
        ufe[i, 1] = (float(r[2]) - 30.0) / 15.0
        ufe[i, 2 + int(r[3])] = 1.0
    aff = (ufe @ rng.standard_normal((ufe.shape[1], gmat.shape[1])).astype(np.float32)) @ gmat.T
    aff = (aff - aff.mean()) / aff.std()
    pop = 1.0 / np.arange(1, len(mids) + 1) ** 0.9
    logp = np.log(pop[rng.permutation(len(mids))])[None, :] + 1.5 * aff
    per_user = np.maximum(20, rng.lognormal(4.6, 0.9, len(uids)).astype(np.int64))
    per_user = np.minimum(per_user, len(mids) // 2)
    per_user = (per_user * (n / per_user.sum())).astype(np.int64).clip(20, len(mids) // 2)
    keys = logp + rng.gumbel(size=logp.shape)
    order = np.argsort(-keys, axis=1)
    rows = []
    for i, (u, c) in enumerate(zip(uids, per_user)):
        c = int(c)
        m = order[i, :c]
        r = np.clip(np.rint(3.1 + 0.9 * aff[i, m] + 0.7 * rng.standard_normal(c)), 1, 5).astype(np.int64)
        t = rng.integers(956703932, 1046454590, size=c)
        rows.append(np.stack([np.full(c, u), mids[m], r, t], axis=1))
    allr = np.concatenate(rows)
    with open(path, "w") as fh:
        fh.write("\n".join("::".join(map(str, row)) for row in allr.tolist()))
        fh.write("\n")


def run_epoch_block(ctx: Ctx):
    """BASELINE config 1 for real: MovieLens-1M (real users.dat / movies.dat, synthesised ratings.dat) through the
    REFERENCE's own loader once on the host, then one full training epoch on the GPU (device feed + CUDA-graph step)
    and the exact top-100 evaluation of every test user on the GPU (item tower -> masked fused top-K -> device
    metrics), checked against the oracle pipeline (numpy towers + np.dot/argsort twin + restated Evaluator) on the same
    weights.  Needs the staged reference loader (baseline/_ref); skipped otherwise."""
    mods = _reference_modules()
    if mods is None:
        return {"skipped": "reference loader not staged (baseline/_ref missing)"}
    import importlib
    import tempfile
    from b200rec.evaluation import Evaluator
    from b200rec.feed import DeviceInteractionFeed
    from b200rec.trainer import TwoTowerTrainer
    from b200rec.training_utils import create_two_tower_model_for_training
    ml = importlib.import_module("src.data.movielens")
    ds_mod = importlib.import_module("src.training.datasets.movielens")
    ref_root = os.path.join(ROOT, "baseline", "_ref", "ml-1m")
    t_host = time.perf_counter()
    with tempfile.TemporaryDirectory() as tmp:
        for f in ("users.dat", "movies.dat"):
            os.symlink(os.path.join(ref_root, f), os.path.join(tmp, f))
        real = os.path.join(ROOT, "ml-1m", "ratings.dat")
        if os.path.exists(real):
            os.symlink(real, os.path.join(tmp, "ratings.dat"))
            ratings_src = "ml-1m/ratings.dat"
        else:
            synth_ratings(os.path.join(tmp, "ratings.dat"), os.path.join(tmp, "users.dat"), os.path.join(tmp, "movies.dat"))
            ratings_src = "synthesised (SURVEY 8c)"
        data = ml.MovieLensLoader(tmp).load_and_preprocess(split_method="time", val_ratio=0.1, test_ratio=0.1,
                                                           implicit_threshold=4.0, min_user_interactions=5,
                                                           min_item_interactions=5)
    train_ds = ds_mod.MovieLensDataset(data.train_interactions, data.users, data.movies, num_negatives=16, is_training=True)
    host_s = time.perf_counter() - t_host
    device = ctx.device
    torch.manual_seed(SEED)
    uf, mf = train_ds.user_features, train_ds.movie_features
    model = create_two_tower_model_for_training(uf.shape[1], mf.shape[1], {"embedding_dim": 128, "hidden_layers": [256, 128],
                                                                            "dropout_rate": 0.2, "temperature": 0.05})
    feed = DeviceInteractionFeed.from_dataset(train_ds, batch_size=1024, shuffle=True, seed=SEED, device=str(device))
    trainer = TwoTowerTrainer(model, feed, [], {"learning_rate": 1e-3, "weight_decay": 1e-5,
                                                "checkpoint_dir": "/tmp/b200rec_bench_ckpt"}, device=str(device))
    trainer.enable_cuda_graph(warm_steps=2)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    loss = trainer.train_epoch(1)
    torch.cuda.synchronize()
    epoch_s = time.perf_counter() - t0
    feed.check()
    # evaluation protocol of scripts/evaluate_model.py:162-234 / Evaluator.evaluate_model
    test = data.test_interactions
    pos_test = test[test["label"] == 1] if "label" in test else test
    gt = {int(u): set(map(int, g)) for u, g in pos_test.groupby("user_idx")["movie_idx"]}
    tr = data.train_interactions
    train_items = {int(u): set(map(int, g)) for u, g in tr.groupby("user_idx")["movie_idx"]}
    test_users = sorted(gt.keys())
    n_items = mf.shape[0]
    ks = [5, 10, 20, 50, 100]
    ev = Evaluator(k_values=ks, num_items=n_items)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    got = ev.evaluate_model(model, test_users, gt, train_items, uf, mf, list(range(n_items)), batch_size=1024, device=str(device))
    torch.cuda.synchronize()
    eval_s = time.perf_counter() - t0
    # oracle pipeline on the same weights (numpy towers -> np.dot + -inf mask + argsort -> restated Evaluator)
    from oracle import metrics as OM
    from oracle.flat_ip import eval_twin_topk
    from oracle.two_tower import TowerOracle
    t0 = time.perf_counter()
    sd = lambda t: {k: v.detach().cpu().numpy() for k, v in t.state_dict().items()}
    ue = TowerOracle(sd(model.user_tower), 2, dtype=np.float32).forward(uf[test_users], training=False)
    ie = TowerOracle(sd(model.item_tower), 2, dtype=np.float32).forward(mf, training=False)
    recs = eval_twin_topk(ue, ie, {u: sorted(v) for u, v in train_items.items()}, test_users, 100)
    want, _ = OM.evaluate({u: recs[u] for u in test_users}, gt, ks, n_items)
    cpu_eval_s = time.perf_counter() - t0
    rows, _ = ev.recommend(model, test_users, train_items, uf, mf, 100, 1024, str(device))
    rows = rows.cpu().numpy()
    exact, _ = OM.evaluate({u: rows[j].tolist() for j, u in enumerate(test_users)}, gt, ks, n_items)
    gd = got.to_dict()
    lists_equal = float(np.mean([rows[j].tolist() == recs[u] for j, u in enumerate(test_users)]))
    # where a list differs from the CPU twin's, is it a score tie?  (north_star: ids exact except at ties within 1e-5)
    with torch.no_grad():
        ue_g = model.get_user_embeddings({"numerical": torch.as_tensor(uf[test_users], dtype=torch.float32).to(device),
                                          "categorical": {}}).cpu().numpy()
        ie_g = model.get_item_embeddings({"numerical": torch.as_tensor(mf, dtype=torch.float32).to(device),
                                          "categorical": {}}).cpu().numpy()
    sc = ue.astype(np.float64) @ ie.astype(np.float64).T
    ok_ties, worst_gap, gaps = 0, 0.0, []
    for j, u in enumerate(test_users):
        a, b = rows[j], np.asarray(recs[u])
        d = a != b
        gap = float(np.abs(sc[j, a[d]] - sc[j, b[d]]).max()) if d.any() else 0.0
        worst_gap = max(worst_gap, gap)
        ok_ties += gap <= 1e-5
        gaps.append(float(np.median(-np.diff(sc[j, b]))))
    tie_diag = {"fraction_of_users_identical_outside_1e-5_ties": ok_ties / max(1, len(test_users)),
                "worst_score_gap_at_a_differing_position": worst_gap,
                "median_gap_between_adjacent_top100_scores": float(np.median(gaps)),
                "max_abs_embedding_diff_gpu_vs_numpy_towers": float(max(np.abs(ue_g - ue).max(), np.abs(ie_g - ie).max()))}
    return {"metric": "train samples/s", "value": len(train_ds) / epoch_s, "unit": "samples/s", "epoch_seconds": epoch_s,
            "train_rows": len(train_ds), "steps": len(feed), "epoch_mean_loss": loss, "ratings": ratings_src,
            "host_preprocessing_seconds": host_s, "eval_seconds": eval_s, "eval_users": len(test_users), "n_items": n_items,
            "metrics": {k: gd[k] for k in ("recall@10", "recall@100", "ndcg@10", "ndcg@100", "hit_rate@10", "mrr", "coverage")},
            "metrics_identical_to_oracle_on_same_lists": bool(all(gd[k] == v for k, v in exact.items())),
            "max_abs_metric_diff_vs_cpu_pipeline": float(max(abs(gd[k] - v) for k, v in want.items())),
            "fraction_of_users_with_identical_top100_list": lists_equal, "list_differences": tie_diag,
            "list_differences_note": "the ML-1M towers see features only: movies with identical genre / year features get "
                                     "identical embeddings, i.e. EXACT score ties, which np.argsort()[::-1] (the CPU twin) "
                                     "and the GPU select (score desc, row asc) order differently; every differing position "
                                     "is such a tie (gap <= 1e-5), which is the north_star's stated exception",
            "cpu_eval_seconds": cpu_eval_s,
            "config": {"workload": "MovieLens-1M two-tower epoch (reference loader on the host once, device feed + CUDA-graph "
                                   "step) + exact top-100 eval of every test user with train-item masking on the GPU"}}


# ------------------------------------------------------------------------------------------------ config 5: serving loop
def run_serve_block(ctx: Ctx, steps: int, warmup: int):
    """BASELINE config 5: user-tower forward on Q users -> 100 M-item x 64-dim bf16 catalogue (row-sharded over the N
    GPUs, 12.8 GB total) -> sharded exact top-1000 -> merge.  Q = 1024 is the headline; a Q sweep shows the HBM-bound
    regime (one catalogue scan serves 1 or 128 queries) that request batching (b200rec.serving.RetrievalBatcher) exploits."""
    from b200rec.dist import ShardedFlatIndex, shard_bounds
    from b200rec.retrieval import FlatIPDeviceIndex
    from b200rec.training_utils import create_two_tower_model_for_training
    device, world, rank = ctx.device, ctx.world, ctx.rank
    NI5, D5, K5, FU = 100_000_000, 64, 1000, 16
    lo, hi = shard_bounds(NI5, world, rank)
    index = FlatIPDeviceIndex(D5, storage="bf16", device=device, row_offset=lo)
    index.add_bf16_rows(make_catalogue_shard(lo, hi, device, NI5, D5, SEED + 5))
    sharded = ShardedFlatIndex.from_device_index(index)
    torch.manual_seed(SEED)
    with torch.device(device):
        model = create_two_tower_model_for_training(FU, FU, {"embedding_dim": D5, "hidden_layers": [128, 64],
                                                              "dropout_rate": 0.2, "temperature": 0.05})
    model.eval()
    pk = _peaks()
    sweep = {}
    out = None
    for Q in (1, 16, 128, 1024):
        feats_host = torch.randn(Q, FU, generator=torch.Generator().manual_seed(SEED + Q)).pin_memory()
        feats = feats_host.to(device)

        def step(i, feats=feats):
            with torch.no_grad():
                emb = model.get_user_embeddings({"numerical": feats, "categorical": {}})
                q_op = index.prepare_queries(emb, normalize=False)
                return sharded.search(q_op, K5)

        ms = timed(ctx, step, steps, max(warmup, 3))
        n_local = hi - lo
        flops = 2.0 * Q * n_local * D5
        bytes_ = n_local * D5 * 2.0 + Q * D5 * 2 + Q * K5 * 12
        t_hbm, t_tc = bytes_ / (pk["hbm_gbs"] * 1e9) * 1e3, flops / (pk["tflops"] * 1e12) * 1e3
        bound = "hbm" if t_hbm >= t_tc else "tensor"
        ach = bytes_ / (ms * 1e-3) / 1e9 if bound == "hbm" else flops / (ms * 1e-3) / 1e12
        peak = pk["hbm_gbs"] if bound == "hbm" else pk["tflops"]
        sweep[str(Q)] = {"ms_per_batch": ms, "qps": Q / ms * 1e3, "bound": bound, "frac": ach / peak,
                         "hbm_floor_ms": t_hbm, "tensor_floor_ms": t_tc}
        if Q == 1024:
            # end to end: host user features -> tower -> sharded search -> host results (this replica's share at N > 1)
            lo_q, hi_q = shard_bounds(Q, world, rank) if world > 1 else (0, Q)
            d_host = torch.empty((hi_q - lo_q, K5), dtype=torch.float32).pin_memory()
            i_host = torch.empty((hi_q - lo_q, K5), dtype=torch.int64).pin_memory()

            def e2e_once():
                f = feats_host.to(device, non_blocking=True)
                with torch.no_grad():
                    emb = model.get_user_embeddings({"numerical": f, "categorical": {}})
                    ds, ii = sharded.search(index.prepare_queries(emb, normalize=False), K5)
                d_host.copy_(ds[lo_q:hi_q], non_blocking=True)
                i_host.copy_(ii[lo_q:hi_q], non_blocking=True)
                torch.cuda.synchronize()

            for _ in range(3):
                e2e_once()
            ctx.barrier()
            t0 = time.perf_counter()
            for _ in range(steps):
                e2e_once()
            ctx.barrier()
            e2e_ms = ctx.max_over_ranks((time.perf_counter() - t0) / steps * 1e3)[0]
            out = {"metric": "top-1000 exact-IP QPS over 100M items (user tower + sharded retrieval)",
                   "value": Q / ms * 1e3, "unit": "queries/s", "ms_per_step": ms, "latency_ms_e2e": e2e_ms,
                   "n_gpus": world, "scaling": "strong", "dtype": "bf16",
                   "config": {"workload": f"user-tower forward ({FU} features -> [128,64] -> {D5}) + exact IP top-{K5} over "
                                          f"{NI5} items x {D5}-dim bf16, query batch {Q}, catalogue row-sharded over {world} GPU(s)"},
                   "e2e": {"value": Q / e2e_ms * 1e3, "unit": "queries/s", "h2d_bytes_per_step": Q * FU * 4 * world,
                           "d2h_bytes_per_step": Q * K5 * 12},
                   "roofline": {"bound": bound, "achieved": ach, "peak": peak, "unit": "GB/s" if bound == "hbm" else "TFLOP/s",
                                "frac": ach / peak, "traffic": None, "scope": "whole serving step (tower + sample + search + merge)",
                                "algorithmic_bytes": bytes_, "flops_per_step": flops, "hbm_floor_ms": t_hbm,
                                "tensor_floor_ms": t_tc, "peak_source": pk["source"]}}
    out["q_sweep"] = sweep
    del sharded, index, model
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------------ main arm
def run_block(extra: dict, world: int, key: str, fn, *a, **kw) -> None:
    """One extra block of the line.  On a single GPU a failing block is recorded as {"error": ...} instead of costing
    the headline (the retrieval numbers are already measured); under torchrun an exception stays fatal, because a rank
    that skipped a block would leave its peers waiting inside that block's collectives."""
    if world > 1:
        extra[key] = fn(*a, **kw)
        return
    try:
        extra[key] = fn(*a, **kw)
    except Exception as exc:  # noqa: BLE001
        import gc
        extra[key] = {"error": repr(exc)[:300]}
        del exc
        gc.collect()
        if torch.cuda.is_available():
            torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-train", action="store_true", help="retrieval only (skip every extra block)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--blocks", default="train,ml1m,epoch,cfg4,serve", help="extra blocks to run (comma separated)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the top-K scores and ids of the last timed search as DIR/topk_scores.npy (float32) and "
                         "DIR/topk_ids.npy (float64), to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU arm (--impl b200)")

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: there is no CPU fallback for the b200rec kernels")
    import torch.distributed as dist
    from b200rec import _native as N
    from b200rec.dist import ShardedFlatIndex, shard_bounds
    from b200rec.retrieval import FlatIPDeviceIndex

    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    ctx = Ctx(device, world, rank)
    warmup = max(args.warmup, 3)
    steps = args.steps
    blocks = set() if args.no_train else {b for b in args.blocks.split(",") if b}
    want_cpu = (not args.no_cpu_baseline) and rank == 0 and world == 1

    lo, hi = shard_bounds(N_ITEMS, world, rank)
    index = FlatIPDeviceIndex(DIM, storage="bf16", device=device, row_offset=lo)
    index.add_bf16_rows(make_catalogue_shard(lo, hi, device))
    sharded = ShardedFlatIndex.from_device_index(index)
    q_host = make_queries_host()
    q_np = q_host.numpy()
    q_op = index.prepare_queries(q_host.pin_memory(), normalize=False)  # resident bf16 operand for the `value` region

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()  # nvidia-smi needs ~100 ms to produce its first line: start it before the warm-up
    for _ in range(warmup):
        s, i = sharded.search(q_op, TOPK)
    ctx.barrier()
    n_before = len(sampler.rows)
    l0 = N.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        s, i = sharded.search(q_op, TOPK)
    e1.record()
    ctx.barrier()
    ms = e0.elapsed_time(e1) / steps
    launches = N.launch_count() - l0
    if args.dump_outputs and rank == 0:
        # what a caller of the timed search received in its last step (ids as float64: exact below 2^53)
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "topk_scores.npy"), s.float().cpu().numpy())
        np.save(os.path.join(args.dump_outputs, "topk_ids.npy"), i.cpu().numpy().astype(np.float64))
    if rank == 0:
        sampler.rows = sampler.rows[n_before:] or sampler.rows[-3:]
    clocks = sampler.stop() if rank == 0 else None
    if world > 1:
        parity = parity_check(ctx, index, q_host, s, i)     # holds collectives: an exception must stay fatal on every rank
    else:
        try:
            parity = parity_check(ctx, index, q_host, s, i)
        except Exception as exc:  # noqa: BLE001 - a checker failure is reported, it does not erase the measurement
            parity = {"queries": 0, "ok": False, "error": repr(exc)[:300]}

    # dominant kernel alone (CUDA events recorded by the library around the fused kernel on its launching stream)
    import ctypes
    lib = N.lib()
    lib.b200rec_debug_topk_kernel_timing.argtypes = [ctypes.c_int, ctypes.POINTER(ctypes.c_float)]
    lib.b200rec_debug_topk_kernel_timing(1, None)
    kms = []
    for _ in range(steps):
        sharded.search(q_op, TOPK)
        out = ctypes.c_float(0)
        lib.b200rec_debug_topk_kernel_timing(1, ctypes.byref(out))
        kms.append(out.value)
    lib.b200rec_debug_topk_kernel_timing(0, None)
    kernel_ms = float(np.mean(kms))

    # end to end through the plugin call: HOST numpy queries -> (D, I) numpy; faiss.normalize_L2 + operand cast on the
    # device; at N > 1 every replica returns its share of the answers (full result on every replica in e2e_sync_call)
    def run_stream(n):
        last = None
        gen = (sharded.search_stream((q_np for _ in range(n)), TOPK, normalize=True, share_results=True) if world > 1
               else index.search_stream((q_np for _ in range(n)), TOPK, normalize=True))
        for last in gen:
            pass
        return last

    run_stream(3)
    ctx.barrier()
    t0 = time.perf_counter()
    d_np, i_np = run_stream(steps)
    ctx.barrier()
    e2e_ms = (time.perf_counter() - t0) / steps * 1e3
    lo_q, hi_q = shard_bounds(N_QUERIES, world, rank) if world > 1 else (0, N_QUERIES)

    def sync_call():
        return sharded.search_numpy(q_np, TOPK, normalize=True) if world > 1 else index.search(q_np, TOPK, normalize=True)

    for _ in range(2):
        d_sync, i_sync = sync_call()
    # the streamed (double-buffered) call and the blocking call share the normalise + cast, so their answers must be
    # identical; the resident-operand path above skipped the (idempotent up to rounding) re-normalisation
    e2e_same = bool(np.array_equal(i_np, np.asarray(i_sync)[lo_q:hi_q] if world > 1 else np.asarray(i_sync)))
    ctx.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        sync_call()
    ctx.barrier()
    sync_ms = (time.perf_counter() - t0) / steps * 1e3
    ms, e2e_ms, kernel_ms, sync_ms = ctx.max_over_ranks(ms, e2e_ms, kernel_ms, sync_ms)

    del sharded, index, q_op, s, i
    torch.cuda.empty_cache()
    extra = {}

    def block(key, fn, *a, **kw):
        run_block(extra, world, key, fn, *a, **kw)

    if "train" in blocks:
        block("train", run_table_train_block, ctx, steps, warmup, want_cpu, name="config 2 (synthetic)", NU=1_000_000,
              NI=100_000, edim=64, hidden=[128, 64], E=64, sparse_tables=False, check_dp=True)
    if "ml1m" in blocks and rank == 0 and world == 1:
        block("train_ml1m", run_ml1m_block, ctx, steps, 20, want_cpu)
    if "epoch" in blocks and rank == 0 and world == 1:
        block("epoch_ml1m", run_epoch_block, ctx)
    if "cfg4" in blocks:
        block("train_cfg4", run_table_train_block, ctx, steps, warmup, False, name="config 4 (synthetic)",
              NU=50_000_000, NI=5_000_000, edim=128, hidden=[256, 128], E=128, sparse_tables=True, check_dp=False)
    if "serve" in blocks:
        block("serve", run_serve_block, ctx, steps, warmup)
    cpu = None
    if want_cpu:
        threads = host_threads()
        rows, queries = 1_000_000, N_QUERIES
        try:
            v, dt, what = cpu_retrieval_baseline(rows, queries, threads)
            cpu = {"value": v, "unit": "queries/s", "cores": threads, "kind": "port",
                   "sample": f"{queries} queries x {rows} rows fp32 ({dt:.2f} s per pass, mean of 3) on {threads} threads, {what}, "
                             f"QPS scaled linearly to {N_ITEMS} rows"}
        except Exception as exc:  # noqa: BLE001 - the measured GPU line must still be printed
            cpu = {"error": repr(exc)[:300]}
    if rank == 0:
        peaks = _peaks()
        traffic = None  # DRAM bytes of one launch of the dominant kernel, from the committed ncu --set full capture
        for name in ("r02_topk_traffic.json", "r01_topk_traffic.json"):
            tpath = os.path.join(ROOT, "profiles", name)
            if world == 1 and os.path.exists(tpath):
                try:
                    with open(tpath) as fh:
                        tj = json.load(fh)
                    traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]
                    break
                except Exception:  # noqa: BLE001 - unreadable capture summary: traffic stays null
                    traffic = None
        n_local = (N_ITEMS + world - 1) // world
        flops = 2.0 * N_QUERIES * n_local * DIM
        achieved = flops / (kernel_ms * 1e-3) / 1e12
        line = {"metric": METRIC, "value": N_QUERIES / ms * 1e3, "unit": "queries/s", "n_gpus": world, "steps": steps,
                "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": primary_config(world),
                "e2e": {"value": N_QUERIES / e2e_ms * 1e3, "unit": "queries/s",
                        "h2d_bytes_per_step": N_QUERIES * DIM * 4 * world, "d2h_bytes_per_step": N_QUERIES * TOPK * 12,
                        "api": "index.search_stream(numpy query batches, k) -> (D, I) numpy per batch (pinned double "
                               "buffering inside the call)", "results_equal_blocking_call": e2e_same},
                "e2e_sync_call": {"value": N_QUERIES / sync_ms * 1e3, "unit": "queries/s",
                                  "api": "index.search(numpy queries, k) -> (D, I) numpy, one blocking call per step"},
                "gpu_launches": int(launches), "parity_checked": parity,
                "clocks": clocks,
                "roofline": {"kernel": "stream_scores2_kernel<2,TopkEpi> (scoring GEMM fused with top-K select)",
                             "bound": "tensor", "achieved": achieved, "peak": peaks["tflops"], "unit": "TFLOP/s",
                             "frac": achieved / peaks["tflops"], "traffic": traffic, "kernel_ms": kernel_ms,
                             "frac_of_burst_peak": achieved / peaks["tflops_burst"],
                             "step_frac": flops / (ms * 1e-3) / 1e12 / peaks["tflops"],
                             "algorithmic_bytes": n_local * DIM * 2 + N_QUERIES * DIM * 2 + N_QUERIES * TOPK * 12,
                             "flops_per_launch": flops, "peak_source": peaks["source"],
                             "hbm_floor_ms": n_local * DIM * 2 / (peaks["hbm_gbs"] * 1e9) * 1e3},
                "cpu_baseline": cpu}
        line.update(extra)
        print(json.dumps(line), flush=True)
    if world > 1:
        import gc
        import threading
        gc.collect()
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        # the line is out; a wedged communicator teardown must not turn a finished run into a timeout
        killer = threading.Timer(60.0, lambda: os._exit(0))
        killer.daemon = True
        killer.start()
        dist.destroy_process_group()
        killer.cancel()


if __name__ == "__main__":
    main()
