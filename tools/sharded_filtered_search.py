"""Row-sharded filtered exact top-K on the config-3 catalogue, G row shards emulated on ONE GPU: each shard's steps (filtered
sample, filtered search from the pooled threshold) run one after another on the same device, so the per-shard device
times are what each of G GPUs would spend; the NVLink / NCCL exchange and the barriers are NOT in these numbers.

Workload: 10 M x 128 bf16 rows built as bench.py builds them (seed 1234), queries = bench.py's, k = 100, G in {2, 8},
Q in {1, 128, 4096}; filters at f in {1, 0.5, 0.05, 0.01}: "uniform" (f * N rows drawn over the whole catalogue) and
"one shard" (f of shard 0's rows, nothing elsewhere: a global fraction of f / G).  Per case, CUDA-event times (median
over alternated repetitions after warm-up), in ms:
  sample[g], search[g]   - per-shard filtered sample / search (compacted operands cached)
  pooled, merge          - the pooled k-th of the G samples, the k-way merge of the G results
  filtered               - max(sample) + pooled + max(search) + merge: the device critical path without the exchange
  filtered_1st           - the same with the compacted operands gathered on first use
  unfiltered             - the same critical path of the unfiltered sharded search, alternated with the above
  single                 - the single-GPU filtered search over the whole catalogue (search_device(sel=))
plus the path each shard took (bitmap / compact / none), whether it contributed a real sample, how far the pooled
threshold lies below the exact k-th allowed score (median over queries), and a parity check: the emulated sharded
result must equal the single-GPU filtered search bit for bit.  Writes one JSON file (--out) with the card, power limit
and SM clock read in the same run.

    python tools/sharded_filtered_search.py --out PATH [--gpus 2 8] [--reps 5]
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
FRACS = (1.0, 0.5, 0.05, 0.01)


class Timer:
    def __init__(self):
        self.ev = []

    def __call__(self, fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        self.ev.append((e0, e1))
        return out

    def read(self):
        torch.cuda.synchronize()
        out = [a.elapsed_time(b) for a, b in self.ev]
        self.ev = []
        return out


def run_sharded(shards, q_op, sels, timer):
    """Emulated sharded search (sels None = unfiltered): per-shard sample, pooled k-th, per-shard search, merge."""
    G = len(shards)
    kx = ShardedFlatIndex.exchange_width(KK, G)
    if sels is None:
        vals = [timer(lambda ix=ix: ix.sample_device(q_op, KK, kx, G)) for ix in shards]
    else:
        vals = [timer(lambda ix=ix, s=s: ix.sample_filtered(q_op, KK, kx, G, s)) for ix, s in zip(shards, sels)]
    v = torch.stack(vals).contiguous()
    tau = timer(lambda: K.topk_pooled_kth(v, KK))
    if sels is None:
        parts = [timer(lambda ix=ix: ix.search_device(q_op, KK, tau_init=tau)) for ix in shards]
    else:
        parts = [timer(lambda ix=ix, s=s: ix.search_filtered_shard(q_op, KK, s, tau)) for ix, s in zip(shards, sels)]
    s_, i_ = torch.stack([p[0] for p in parts]).contiguous(), torch.stack([p[1] for p in parts]).contiguous()
    out = timer(lambda: K.topk_merge(s_, i_, KK))
    return out, tau, v


def split(ms, G):
    sample, pooled, search, merge = ms[:G], ms[G], ms[G + 1: 2 * G + 1], ms[2 * G + 1]
    return {"sample": sample, "pooled": pooled, "search": search, "merge": merge,
            "critical": max(sample) + pooled + max(search) + merge}


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
    full = FlatIPDeviceIndex(bench.DIM, storage="bf16", device=dev)
    full.add_bf16_rows(cat)
    N = full.ntotal
    q_all = bench.make_queries_host()
    rng = np.random.default_rng(bench.SEED)
    cases = []
    for G in args.gpus:
        shards = []
        for g in range(G):
            lo, hi = shard_bounds(N, G, g)
            ix = FlatIPDeviceIndex(bench.DIM, storage="bf16", device=dev, row_offset=lo)
            ix.add_bf16_rows(cat[lo:hi])
            shards.append(ix)
        lo0, hi0 = shard_bounds(N, G, 0)
        filters = []
        for f in FRACS:
            filters.append(("uniform", f, np.sort(rng.permutation(N)[: int(round(f * N))]) if f < 1 else np.arange(N)))
            n0 = int(round(f * (hi0 - lo0)))
            filters.append(("one shard", f, np.sort(lo0 + rng.permutation(hi0 - lo0)[:n0]) if f < 1 else np.arange(lo0, hi0)))
        for kind, f, rows in filters:
            sels = [ix.row_filter(rows=shard_filter_rows(ix.row_offset, ix.ntotal, rows=rows)) for ix in shards]
            fsel = full.row_filter(rows=rows)
            for Q in QS:
                q_op = full.prepare_queries(q_all[:Q].to(dev), normalize=False)
                timer = Timer()
                for _ in range(2):                                                   # warm-up of every shape
                    run_sharded(shards, q_op, sels, timer)
                    run_sharded(shards, q_op, None, timer)
                    full.search_device(q_op, KK, sel=fsel)
                timer.read()
                res = {"filtered": [], "filtered_1st": [], "unfiltered": [], "single": []}
                for _ in range(args.reps):                                           # alternated
                    for s in sels:
                        s._compact = None
                    run_sharded(shards, q_op, sels, timer)
                    res["filtered_1st"].append(split(timer.read(), G))
                    (d, i), tau, vals = run_sharded(shards, q_op, sels, timer)
                    res["filtered"].append(split(timer.read(), G))
                    run_sharded(shards, q_op, None, timer)
                    res["unfiltered"].append(split(timer.read(), G))
                    sd, si = timer(lambda: full.search_device(q_op, KK, sel=fsel))
                    res["single"].append(timer.read()[0])
                parity = bool(torch.equal(d, sd) and torch.equal(i, si))
                kth = sd[:, KK - 1].float()
                gap = (kth - tau).cpu().numpy()
                med = lambda xs: float(np.median(xs))   # noqa: E731
                case = {"G": G, "filter": kind, "f": f, "n_allowed": int(sum(s.n_allowed for s in sels)), "Q": Q,
                        "k": KK, "reps": args.reps,
                        "paths": ["none" if s.n_allowed == 0 else
                                  ("compact" if s.fraction < FlatIPDeviceIndex.FILTER_COMPACT_BELOW else "bitmap")
                                  for s in sels],
                        "sampled": [bool((vals[g] > -3.0e38).any()) for g in range(G)],
                        "bound_gap_median": float(np.median(gap)) if np.isfinite(gap).all() else None,
                        "no_pruning_queries": int((tau.cpu().numpy() <= -3.0e38).sum()),
                        "ms": {"filtered": med([r["critical"] for r in res["filtered"]]),
                               "filtered_1st": med([r["critical"] for r in res["filtered_1st"]]),
                               "unfiltered": med([r["critical"] for r in res["unfiltered"]]),
                               "single": med(res["single"]),
                               "filtered_sample_per_shard": [med([r["sample"][g] for r in res["filtered"]]) for g in range(G)],
                               "filtered_search_per_shard": [med([r["search"][g] for r in res["filtered"]]) for g in range(G)],
                               "pooled": med([r["pooled"] for r in res["filtered"]]),
                               "merge": med([r["merge"] for r in res["filtered"]])},
                        "parity_equals_single_gpu_filtered": parity}
                cases.append(case)
                print(json.dumps({k: case[k] for k in ("G", "filter", "f", "Q", "paths", "parity_equals_single_gpu_filtered")}
                                 | {"ms": {k: round(v, 3) for k, v in case["ms"].items() if not isinstance(v, list)}}),
                      flush=True)
                del q_op
            for s in sels + [fsel]:
                s._compact = None
            del sels, fsel
            torch.cuda.empty_cache()
        del shards
    result = {"tool": "tools/sharded_filtered_search.py",
              "workload": "10M x 128 bf16 (bench.py catalogue, seed 1234), k = 100, G row shards emulated on one GPU "
                          "(exchange and barriers not included)",
              "card_before": card_before, "card_after": smi(), "seconds": round(time.time() - t_start, 1),
              "filter_compact_below": FlatIPDeviceIndex.FILTER_COMPACT_BELOW, "cases": cases,
              "all_parity_ok": all(c["parity_equals_single_gpu_filtered"] for c in cases)}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps({"all_parity_ok": result["all_parity_ok"], "card": result["card_after"]}))
    sys.exit(0 if result["all_parity_ok"] else 1)


if __name__ == "__main__":
    main()
