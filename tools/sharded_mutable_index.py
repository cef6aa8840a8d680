"""Live catalogue on the row-sharded index, config-3 catalogue, G row shards emulated on ONE GPU: each shard's steps
(sample_shard, search_shard from the pooled threshold) run one after another on the same device, so the per-shard device
times are what each of G GPUs would spend; the NVLink / NCCL exchange and the barriers are NOT in these numbers.

Workload: 10 M x 128 bf16 rows built as bench.py builds them (seed 1234), queries = bench.py's, k = 100, G in {2, 8},
Q in {1, 128, 4096}.  Removed rows: a fraction r in {0.0001, 0.01, 0.1, 0.5} of the catalogue drawn uniformly
("uniform"), or the fraction r of shard 0's rows with nothing removed elsewhere ("one shard").  One filtered case: a
uniform filter of f = 0.5 (every shard takes the compact path) with 1 % of the rows removed uniformly.  Per case,
CUDA-event times (median over alternated repetitions after warm-up), in ms, of the device critical path
max(shard sample) + pooled k-th + max(shard search) + merge:
  unmutated   - the sharded step over the same shards with nothing removed
  mutated     - the sharded step with the rows removed
  compacted   - the same after every shard ran compact()
  single      - the single-GPU search over the same mutated catalogue (search_device)
plus the per-shard sample / search times of the mutated step and a parity check: the mutated sharded result must
equal the single-GPU mutated search bit for bit, and the compacted one the mutated one mapped through the old -> new
row map.  Also timed (host wall clock around work that ends in a device synchronise): every shard's compact() and an
update_rows of 10 K host rows per shard.  Writes one JSON file (--out) with the card, power limit and SM clock read in
the same run.

    python tools/sharded_mutable_index.py --out PATH [--gpus 2 8] [--reps 5]
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench  # noqa: E402  (catalogue / query generators of the benchmark)
from filtered_search import smi  # noqa: E402
from b200rec import kernels as K  # noqa: E402
from b200rec.dist import ShardedFlatIndex, shard_bounds, shard_filter_rows  # noqa: E402
from b200rec.retrieval import FlatIPDeviceIndex  # noqa: E402

KK = 100
QS = (1, 128, 4096)
REMOVED = (0.0001, 0.01, 0.1, 0.5)


class Timer:
    def __init__(self):
        self.ev = []

    def __call__(self, label, fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        self.ev.append((label, e0, e1))
        return out

    def read(self):
        torch.cuda.synchronize()
        out = {}
        for label, a, b in self.ev:
            out.setdefault(label, []).append(a.elapsed_time(b))
        self.ev = []
        return out


def run_sharded(shards, q_op, sels, timer):
    """Emulated sharded step: per-shard sample, pooled k-th (no threshold when an unmutated, unfiltered shard has no
    sampling pass: the agreement round of the real exchange), per-shard search, merge."""
    G = len(shards)
    kx = ShardedFlatIndex.exchange_width(KK, G)
    sels = sels or [None] * G
    vals = [timer("sample", lambda ix=ix, s=s: ix.sample_shard(q_op, KK, kx, G, sel=s)) for ix, s in zip(shards, sels)]
    tau = None
    if all(v is not None for v in vals):
        v = torch.stack(vals).contiguous()
        tau = timer("pooled", lambda: K.topk_pooled_kth(v, KK))
    parts = [timer("search", lambda ix=ix, s=s: ix.search_shard(q_op, KK, tau, sel=s)) for ix, s in zip(shards, sels)]
    s_, i_ = torch.stack([p[0] for p in parts]).contiguous(), torch.stack([p[1] for p in parts]).contiguous()
    return timer("merge", lambda: K.topk_merge(s_, i_, KK))


def critical(ms):
    return max(ms["sample"]) + sum(ms.get("pooled", [0.0])) + max(ms["search"]) + ms["merge"][0]


def make_shards(cat, G, dev):
    """G shards over the rows of `cat` without a copy (each takes over its contiguous slice)."""
    shards = []
    for g in range(G):
        lo, hi = shard_bounds(cat.shape[0], G, g)
        ix = FlatIPDeviceIndex(bench.DIM, storage="bf16", device=dev, row_offset=lo)
        ix.add_bf16_rows(cat[lo:hi])
        shards.append(ix)
    return shards


def remove(shards, single, rows):
    for ix in shards:
        ix.remove_rows(shard_filter_rows(ix.row_offset, ix.ntotal, rows=rows))
    single.remove_rows(rows)


def compact(shards):
    """Every shard's compact() (host wall clock, ending in a synchronise) and the global old -> new map."""
    secs, maps, off = [], [], 0
    for ix in shards:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        local = ix.compact()
        torch.cuda.synchronize()
        secs.append(time.perf_counter() - t0)
        maps.append(np.where(local >= 0, local + off, -1))
        ix.row_offset = off
        off += ix.ntotal
    return np.concatenate(maps), secs


def measure(columns, q_op, reps, timer):
    """columns: name -> callable(timer) -> result.  Warm-up twice, then `reps` alternated rounds; (medians, results)."""
    for _ in range(2):
        for fn in columns.values():
            fn(timer)
    timer.read()
    got, out = {name: [] for name in columns}, {}
    for _ in range(reps):
        for name, fn in columns.items():
            out[name] = fn(timer)
            got[name].append(timer.read())
    med = lambda xs: float(np.median(xs))   # noqa: E731
    ms = {name: med([critical(r) if "sample" in r else r["single"][0] for r in rs]) for name, rs in got.items()}
    m = got["mutated"]
    ms["mutated_sample_per_shard"] = [med([r["sample"][g] for r in m]) for g in range(len(m[0]["sample"]))]
    ms["mutated_search_per_shard"] = [med([r["search"][g] for r in m]) for g in range(len(m[0]["search"]))]
    return ms, out


def run_case(G, kind, r, removed, base, mutated, single, q_all, dev, reps, sel_rows=None):
    """One removal state over every Q: unmutated / mutated / single columns, then compact() and the compacted column."""
    def sels_of(shards, rows):
        if rows is None:
            return None
        return [ix.row_filter(rows=shard_filter_rows(ix.row_offset, ix.ntotal, rows=rows)) for ix in shards]
    base_sels, mut_sels = sels_of(base, sel_rows), sels_of(mutated, sel_rows)
    single_sel = None if sel_rows is None else single.row_filter(rows=sel_rows)
    remove(mutated, single, removed)
    timer = Timer()
    cases, kept = [], {}
    for Q in QS:
        q_op = single.prepare_queries(q_all[:Q].to(dev), normalize=False)
        cols = {"unmutated": lambda t: run_sharded(base, q_op, base_sels, t),
                "mutated": lambda t: run_sharded(mutated, q_op, mut_sels, t),
                "single": lambda t: t("single", lambda: single.search_device(q_op, KK, sel=single_sel))}
        ms, out = measure(cols, q_op, reps, timer)
        parity = bool(torch.equal(out["mutated"][0], out["single"][0]) and torch.equal(out["mutated"][1], out["single"][1]))
        kept[Q] = (q_op, out["mutated"])
        cases.append({"G": G, "removed": kind, "r": r, "n_removed": int(np.unique(removed).size), "Q": Q, "k": KK,
                      "filter": None if sel_rows is None else {"kind": "uniform", "f": 0.5}, "reps": reps, "ms": ms,
                      "paths": [("bitmap" if s.fraction >= FlatIPDeviceIndex.FILTER_COMPACT_BELOW else "compact")
                                for s in mut_sels] if mut_sels else None,
                      "sampling_pass": [ix.has_sample_pass(Q, KK) for ix in mutated],
                      "parity_mutated_equals_single_gpu": parity})
    remap, secs = compact(mutated)
    comp_sels = sels_of(mutated, None if sel_rows is None else np.unique(remap[sel_rows][remap[sel_rows] >= 0]))
    for case in cases:
        q_op, (md, mi) = kept[case["Q"]]
        ms, out = measure({"mutated": lambda t: run_sharded(mutated, q_op, comp_sels, t)}, q_op, reps, timer)
        case["ms"]["compacted"] = ms["mutated"]
        want = torch.from_numpy(np.where(mi.cpu().numpy() >= 0, remap[np.maximum(mi.cpu().numpy(), 0)], -1)).to(dev)
        case["parity_compacted_equals_mutated_mapped"] = bool(torch.equal(out["mutated"][0], md)
                                                              and torch.equal(out["mutated"][1], want))
        case["compact_s_per_shard"] = secs
        print(json.dumps({k: case[k] for k in ("G", "removed", "r", "Q", "parity_mutated_equals_single_gpu",
                                               "parity_compacted_equals_mutated_mapped")}
                         | {"ms": {k: round(v, 3) for k, v in case["ms"].items() if not isinstance(v, list)}}), flush=True)
    return cases


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="JSON file to write")
    ap.add_argument("--gpus", type=int, nargs="+", default=[2, 8])
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    dev = torch.device("cuda", torch.cuda.current_device())
    card_before = smi()
    t_start = time.time()
    cat = bench.make_catalogue_shard(0, bench.N_ITEMS, dev)
    N = cat.shape[0]
    q_all = bench.make_queries_host()
    rng = np.random.default_rng(bench.SEED)
    cases, updates = [], []
    for G in args.gpus:
        base = make_shards(cat, G, dev)
        lo0, hi0 = shard_bounds(N, G, 0)
        states = []
        for r in REMOVED:
            states.append(("uniform", r, rng.permutation(N)[: int(round(r * N))], None))
            states.append(("one shard", r, lo0 + rng.permutation(hi0 - lo0)[: int(round(r * (hi0 - lo0)))], None))
        states.append(("uniform", 0.01, rng.permutation(N)[: N // 100], np.sort(rng.permutation(N)[: N // 2])))
        for kind, r, removed, sel_rows in states:
            mutated = make_shards(cat, G, dev)
            single = FlatIPDeviceIndex(bench.DIM, storage="bf16", device=dev)
            single.add_bf16_rows(cat)
            cases += run_case(G, kind, r, removed, base, mutated, single, q_all, dev, args.reps, sel_rows)
            del mutated, single
            torch.cuda.empty_cache()
        # update_rows of 10 K host rows per shard, written with the values the rows hold (the shared catalogue stays)
        secs = []
        for _ in range(1 + args.reps):
            per = []
            for ix in base:
                rows = np.sort(rng.permutation(ix.ntotal)[:10_000])
                x = ix._cat[torch.from_numpy(rows).to(dev), : bench.DIM].float().cpu().numpy()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                ix.update_rows(rows, x)
                torch.cuda.synchronize()
                per.append(time.perf_counter() - t0)
            secs.append(per)
        updates.append({"G": G, "rows_per_shard": 10_000, "ms_per_shard_median":
                        [float(np.median([s[g] for s in secs[1:]])) * 1e3 for g in range(G)]})
        del base
        torch.cuda.empty_cache()
    result = {"tool": "tools/sharded_mutable_index.py",
              "workload": "10M x 128 bf16 (bench.py catalogue, seed 1234), k = 100, G row shards emulated on one GPU "
                          "(exchange and barriers not included)",
              "card_before": card_before, "card_after": smi(), "seconds": round(time.time() - t_start, 1),
              "cases": cases, "update_rows": updates,
              "all_parity_ok": all(c["parity_mutated_equals_single_gpu"] and c["parity_compacted_equals_mutated_mapped"]
                                   for c in cases)}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps({"all_parity_ok": result["all_parity_ok"], "card": result["card_after"], "update_rows": updates}))
    sys.exit(0 if result["all_parity_ok"] else 1)


if __name__ == "__main__":
    main()
