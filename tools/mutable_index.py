"""Mutable catalogue on the config-3 catalogue: what update_rows / remove_rows / compact() cost, and what removed rows
cost the search, in one process.

Workload: 10 M x 128 bf16 rows built as bench.py builds them (seed 1234), bench.py's queries, k = 100, Q in {1, 128, 4096}.
  search      - per dead fraction (0.01 %, 1 %, 10 %, 50 % of the rows removed at random): the search over the live rows
                (live bitmap inside the fused kernel, masked sampling pass), the unmutated index and the same index after
                compact(), CUDA-event ms per call, median over alternated repetitions after warm-up; remove_rows and
                compact() times for that fraction
  update_rows - batches of 1 / 1 K / 100 K rows: device time of the fused normalise + cast + scatter launch (rows already
                on the device) against its HBM floor rows * (4 d read + 2 ld written) bytes at 7.7 TB/s, and the
                end-to-end call from host numpy (host clock around the call and a synchronise)
  patch       - one b200rec_patch_compacted launch (10 K changed rows) on a cached compacted filter with f = 0.5, update
                and removal, next to a first gather of that filter
  steady      - 4096-query search + a 10 K-row update batch (device-resident rows) per step against the search alone, on
                an index with 1 % of its rows removed
Parity: the first 32 queries of every mutated search against the oracle over the live rows (bf16 rows upcast to fp32,
ids mapped back); the compacted index's answers mapped back through the returned row map equal the masked search's.
Writes one JSON file (--out) with the card, power limit and SM clock read in the same run.

    python tools/mutable_index.py --out PATH [--reps 5]
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
from b200rec import kernels as KK  # noqa: E402
from b200rec.retrieval import FlatIPDeviceIndex  # noqa: E402
from filtered_search import oracle, parity, smi, timed  # noqa: E402

K = 100
QS = (1, 128, 4096)
DEAD = (1e-4, 1e-2, 0.1, 0.5)
N_CHECK = 32
HBM = 7.7e12


def clone(index):
    c = FlatIPDeviceIndex(index.d, storage="bf16", device=index.device)
    c.add_bf16_rows(index._cat[: index.ntotal].clone())
    return c


def med(v):
    return float(np.median(v))


def alternate(fns, reps):
    for fn in fns.values():
        fn()
    torch.cuda.synchronize()
    times = {p: [] for p in fns}
    outs = {}
    for _ in range(reps):
        for p, fn in fns.items():
            ms, out = timed(fn)
            times[p].append(ms)
            outs[p] = out
    return {p: med(v) for p, v in times.items()}, outs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="JSON file to write")
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    dev = torch.device("cuda", torch.cuda.current_device())
    card_before = smi()
    t_start = time.time()
    base = FlatIPDeviceIndex(bench.DIM, storage="bf16", device=dev)
    base.add_bf16_rows(bench.make_catalogue_shard(0, bench.N_ITEMS, dev))
    N, d, ld = base.ntotal, base.d, base.ld
    q_all = bench.make_queries_host()
    qs_check = q_all[:N_CHECK].to(torch.bfloat16).to(torch.float32).numpy()
    q_ops = {Q: base.prepare_queries(q_all[:Q].to(dev)) for Q in QS}
    rng = np.random.default_rng(bench.SEED)
    result = {"tool": "tools/mutable_index.py", "workload": "10M x 128 bf16 (bench.py catalogue, seed 1234), k = 100",
              "card_before": card_before, "search": [], "update_rows": [], "patch": {}, "steady": {}}

    # ---------------------------------------------------------------- search against the dead fraction
    for f in DEAD:
        mut = clone(base)
        dead = np.sort(rng.permutation(N)[: int(round(f * N))])
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ms_rm, n_rm = timed(lambda: mut.remove_rows(dead))
        host_rm = (time.perf_counter() - t0) * 1e3
        live = np.ones(N, bool)
        live[dead] = False
        want = oracle(mut, qs_check, np.flatnonzero(live))
        comp = clone(mut)
        comp._live_bits, comp._live_host, comp._n_dead = mut._live_bits.clone(), mut._live_host.copy(), mut._n_dead
        ms_compact, remap = timed(comp.compact)
        keep = np.flatnonzero(live)
        for Q in QS:
            q = q_ops[Q]
            ms, outs = alternate({"unmutated": lambda: base.search_device(q, K), "live_bitmap": lambda: mut.search_device(q, K),
                                  "after_compact": lambda: comp.search_device(q, K)}, args.reps)
            nq = min(Q, N_CHECK)
            md, mi = (t[:nq].cpu().numpy() for t in outs["live_bitmap"])
            cd, ci = (t[:nq].cpu().numpy() for t in outs["after_compact"])
            check = parity((md, mi), (want[0][:nq], want[1][:nq]))
            mapped = np.where(ci >= 0, keep[np.maximum(ci, 0)], -1)
            case = {"dead_fraction": f, "n_live": mut.n_live, "Q": Q, "ms": ms,
                    "live_bitmap_over_unmutated": ms["live_bitmap"] / ms["unmutated"],
                    "parity": {**check, "compact_equals_masked": bool(np.array_equal(mapped, mi) and np.array_equal(cd, md))}}
            result["search"].append(case)
            print(json.dumps({k: case[k] for k in ("dead_fraction", "Q", "ms")}), flush=True)
        result["search"].append({"dead_fraction": f, "remove_rows": {"rows": int(n_rm), "device_ms": ms_rm,
                                                                      "host_ms": host_rm},
                                 "compact": {"device_ms": ms_compact, "rows_kept": int(keep.size)}})
        del mut, comp
        torch.cuda.empty_cache()

    # ---------------------------------------------------------------- update_rows
    upd = clone(base)
    upd.remove_rows([0])                                  # live bitmap present: the launch also sets the bits
    for n in (1, 1000, 100_000):
        rows = np.sort(rng.choice(N, size=n, replace=False))
        x = rng.standard_normal((n, d)).astype(np.float32)
        rows_dev, x_dev = torch.from_numpy(rows).to(dev), torch.from_numpy(x).to(dev)
        dev_ms = []
        host_ms = []
        for _ in range(args.reps + 1):
            ms, _ = timed(lambda: KK.update_rows(x_dev, rows_dev, upd._cat, upd.kpad, upd.terms, None, upd._live_bits, True))
            dev_ms.append(ms)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            upd.update_rows(rows, x, normalize=True)
            torch.cuda.synchronize()
            host_ms.append((time.perf_counter() - t0) * 1e3)
        floor_ms = n * (4 * d + 2 * ld) / HBM * 1e3
        dms = med(dev_ms[1:])
        result["update_rows"].append({"rows": n, "device_ms": dms, "rows_per_s": n / dms * 1e3, "hbm_floor_ms": floor_ms,
                                      "floor_share": floor_ms / dms, "end_to_end_from_numpy_ms": med(host_ms[1:])})
        print(json.dumps(result["update_rows"][-1]), flush=True)

    # ---------------------------------------------------------------- patch of a cached compacted filter
    sel = upd.row_filter(rows=np.sort(rng.permutation(N)[: N // 2]))
    ms_gather, _ = timed(sel.compacted)
    changed = torch.from_numpy(np.sort(rng.choice(N, size=10_000, replace=False))).to(dev)
    sel._compact_bits = torch.full(((sel.n_allowed + 31) // 32,), -1, dtype=torch.int32, device=dev)
    pu, pr = [], []
    for _ in range(args.reps + 1):
        pu.append(timed(lambda: KK.patch_compacted(changed, sel.rows, upd._cat, sel._compact, sel._compact_bits, True))[0])
        pr.append(timed(lambda: KK.patch_compacted(changed, sel.rows, None, None, sel._compact_bits, False))[0])
    sel0 = base.row_filter(rows=sel.rows.cpu().numpy())          # the same filter on an index without removed rows
    ms_gather0, _ = timed(sel0.compacted)
    result["patch"] = {"filter_f": sel.fraction, "changed_rows": 10_000, "update_ms": med(pu[1:]),
                       "removal_ms": med(pr[1:]), "first_gather_ms": ms_gather,
                       "first_gather_ms_no_removed_rows": ms_gather0}
    del sel0
    print(json.dumps(result["patch"]), flush=True)
    del sel
    torch.cuda.empty_cache()

    # ---------------------------------------------------------------- steady state
    upd.remove_rows(np.sort(rng.permutation(N)[: N // 100]))
    q = q_ops[4096]
    rows_dev = [torch.from_numpy(np.sort(rng.choice(N, size=10_000, replace=False))).to(dev) for _ in range(4)]
    xs = [torch.randn((10_000, d), device=dev) for _ in range(4)]
    steps = 20

    def search_only():
        for _ in range(steps):
            upd.search_device(q, K)

    def search_and_update():
        for s in range(steps):
            upd.search_device(q, K)
            KK.update_rows(xs[s % 4], rows_dev[s % 4], upd._cat, upd.kpad, upd.terms, None, upd._live_bits, True)
    ms, _ = alternate({"search_only": search_only, "search_plus_10k_update": search_and_update}, max(2, args.reps // 2))
    result["steady"] = {"Q": 4096, "dead_fraction": upd._n_dead / N, "steps": steps,
                        "ms_per_step": {p: v / steps for p, v in ms.items()},
                        "overhead": ms["search_plus_10k_update"] / ms["search_only"] - 1.0}
    print(json.dumps(result["steady"]), flush=True)

    # ---------------------------------------------------------------- remove_rows on an index that already has removed rows
    for n in (1, 1000, 100_000):
        host_ms = []
        for _ in range(args.reps + 1):
            rows = rng.choice(N, size=n, replace=False)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            upd.remove_rows(rows)
            torch.cuda.synchronize()
            host_ms.append((time.perf_counter() - t0) * 1e3)
            upd.update_rows(rows, rng.standard_normal((n, d)).astype(np.float32), normalize=True)
        result.setdefault("remove_rows_warm", []).append({"rows": n, "end_to_end_ms": med(host_ms[1:])})
        print(json.dumps(result["remove_rows_warm"][-1]), flush=True)

    result["card_after"] = smi()
    result["seconds"] = round(time.time() - t_start, 1)
    result["all_parity_ok"] = all(c["parity"]["ok"] and c["parity"]["compact_equals_masked"]
                                  for c in result["search"] if "parity" in c)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps({"all_parity_ok": result["all_parity_ok"], "card": result["card_after"]}))


if __name__ == "__main__":
    main()
