"""Filtered exact top-K on the config-3 catalogue: both execution paths of FlatIPDeviceIndex's row filter against the
unfiltered search, in one process, alternated.

Workload: 10 M x 128 bf16 rows built as bench.py builds them (seed 1234), queries = bench.py's, k = 100, Q in
{1, 128, 4096}; filters: uniformly drawn rows at f in {1, 0.5, 0.2, 0.05, 0.01, 0.001} plus one contiguous range.
Per case, CUDA-event times (ms per call, median over alternated repetitions after warm-up) of
  bitmap      - row bitmap tested inside the fused kernel (masked sampling pass)
  compact_1st - compacted catalogue, first use: row gather + search + id remap
  compact     - compacted catalogue, cached
  selected    - what search_device(sel=) picks (FILTER_COMPACT_BELOW)
  unfiltered  - the plain search
and a parity check: the first min(Q, 32) queries re-searched by the oracle over the allowed rows alone (bf16 rows
upcast to fp32, ids mapped back), for every path.  Writes one JSON file (--out) with the card, power limit and SM clock
read in the same run.

    python tools/filtered_search.py --out PATH [--reps 5]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (catalogue / query generators of the benchmark)
from b200rec.retrieval import FlatIPDeviceIndex  # noqa: E402
from oracle.flat_ip import IndexFlatIP, merge_topk  # noqa: E402

K = 100
QS = (1, 128, 4096)
FRACS = (1.0, 0.5, 0.2, 0.05, 0.01, 0.001)
N_CHECK = 32


def smi():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout
        name, pl, sm, smax = [c.strip() for c in out.strip().split(",")]
        return {"name": name, "power_limit_w": float(pl), "sm_mhz": float(sm), "sm_max_mhz": float(smax)}
    except Exception as exc:  # noqa: BLE001
        return {"error": repr(exc)[:200]}


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1), out


def oracle(index, qs, rows):
    """Exact top-k of the first queries over the allowed rows (ascending): the oracle searches those rows alone, in 1 M-row
    chunks of the bf16 rows upcast to fp32, and the ids are mapped back through `rows` (order kept)."""
    run_s = np.full((qs.shape[0], K), -np.finfo(np.float32).max, np.float32)
    run_i = np.full((qs.shape[0], K), -1, np.int64)
    chunk = 1 << 20
    rows_dev = torch.from_numpy(rows).to(index.device)
    for c0 in range(0, rows.size, chunk):
        part = rows[c0:c0 + chunk]
        ix = IndexFlatIP(index.d, db_block=1 << 17)
        ix.add(index._cat[rows_dev[c0:c0 + chunk], : index.d].float().cpu().numpy())
        s, i = ix.search(qs, K)
        run_s, run_i = merge_topk([run_s, s], [run_i, np.where(i >= 0, part[np.maximum(i, 0)], -1)], K)
    return run_s, run_i


def parity(got, want):
    (gs, gi), (ws, wi) = got, want
    diff = gi != wi
    ties_ok = bool((np.abs(gs - ws)[diff] <= 1e-5).all())
    return {"ok": bool(np.allclose(gs, ws, atol=2e-5, rtol=0) and ties_ok and diff.mean() <= 0.01),
            "ids_differing_inside_ties": int(diff.sum()), "max_abs_score_diff": float(np.abs(gs - ws).max())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="JSON file to write")
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    dev = torch.device("cuda", torch.cuda.current_device())
    card_before = smi()
    t_start = time.time()
    index = FlatIPDeviceIndex(bench.DIM, storage="bf16", device=dev)
    index.add_bf16_rows(bench.make_catalogue_shard(0, bench.N_ITEMS, dev))
    N = index.ntotal
    q_all = bench.make_queries_host()
    qs_check = q_all[:N_CHECK].to(torch.bfloat16).to(torch.float32).numpy()
    rng = np.random.default_rng(bench.SEED)
    filters = [(f"uniform f={f:g}", np.sort(rng.permutation(N)[: int(round(f * N))]) if f < 1 else np.arange(N))
               for f in FRACS]
    lo = 3 * N // 10
    filters.append(("contiguous rows [3M, 3.5M) f=0.05", np.arange(lo, lo + N // 20)))
    cases = []
    for fname, rows in filters:
        want = oracle(index, qs_check, rows)
        sel = index.row_filter(rows=rows)
        for Q in QS:
            q_op = index.prepare_queries(q_all[:Q].to(dev), normalize=False)
            paths = {
                "unfiltered": lambda: index.search_device(q_op, K),
                "bitmap": lambda: index._search_filtered(q_op, K, sel, compact=False),
                "compact_1st": lambda: (setattr(sel, "_compact", None), index._search_filtered(q_op, K, sel, compact=True))[1],
                "compact": lambda: index._search_filtered(q_op, K, sel, compact=True),
                "selected": lambda: index.search_device(q_op, K, sel=sel),
            }
            for fn in paths.values():                                        # warm-up of every shape
                fn()
            torch.cuda.synchronize()
            t_bitmap, _ = timed(paths["bitmap"])
            reps = args.reps if t_bitmap < 200 else 2
            times = {p: [] for p in paths}
            outs = {}
            for _ in range(reps):                                            # alternated
                for p, fn in paths.items():
                    ms, out = timed(fn)
                    times[p].append(ms)
                    outs[p] = out
            nq = min(Q, N_CHECK)
            checks = {p: parity(tuple(t[:nq].cpu().numpy() for t in outs[p]), (want[0][:nq], want[1][:nq]))
                      for p in ("bitmap", "compact", "selected")}
            case = {"filter": fname, "f": sel.fraction, "n_allowed": sel.n_allowed, "Q": Q, "k": K, "reps": reps,
                    "selected_path": "compact" if sel.fraction < index.FILTER_COMPACT_BELOW else "bitmap",
                    "ms": {p: float(np.median(v)) for p, v in times.items()},
                    "ms_all": {p: [round(x, 4) for x in v] for p, v in times.items()},
                    "parity": {"queries": nq, "ok": all(c["ok"] for c in checks.values()), "per_path": checks}}
            cases.append(case)
            print(json.dumps({k: case[k] for k in ("filter", "Q", "ms")}), flush=True)
            del q_op
        sel._compact = None
        del sel
        torch.cuda.empty_cache()
    result = {"tool": "tools/filtered_search.py", "workload": "10M x 128 bf16 (bench.py catalogue, seed 1234), k = 100",
              "card_before": card_before, "card_after": smi(), "seconds": round(time.time() - t_start, 1),
              "filter_compact_below": FlatIPDeviceIndex.FILTER_COMPACT_BELOW, "cases": cases,
              "all_parity_ok": all(c["parity"]["ok"] for c in cases)}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps({"all_parity_ok": result["all_parity_ok"], "card": result["card_after"]}))


if __name__ == "__main__":
    main()
