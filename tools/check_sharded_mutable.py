"""torchrun --nproc-per-node G tools/check_sharded_mutable.py : row-sharded search over a MUTATED catalogue == single-GPU
search over the same mutated rows, bit for bit (PEER=1: peer-memory fan-out exchange, PEER=0: NCCL all-gather).  Every
rank passes the same global-row calls: updates straddling the shard boundaries with duplicates, uniform removals, all
but 500 rows of the last shard removed (it keeps no sampling pass once compacted), revived slots, compact() (the same
global map on every rank and on the single index; filters built before are rejected).  Covers unfiltered and filtered
search (bitmap and compact shard paths), search_numpy and n_live().  Exits non-zero on any mismatch."""
import os, sys, numpy as np, torch, torch.distributed as dist
sys.path.insert(0, ".")
from b200rec.dist import ShardedFlatIndex, shard_bounds
from b200rec.retrieval import FlatIPDeviceIndex
rank, world, lr = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(lr); dev = torch.device("cuda", lr)
dist.init_process_group("nccl", device_id=dev)
N, Q, D = int(os.environ.get("NROWS", 2_000_000)), int(os.environ.get("NQ", 4096)), 128
g = torch.Generator(device=dev).manual_seed(7)
cat = torch.nn.functional.normalize(torch.randn(N, D, device=dev, generator=g), dim=1).to(torch.bfloat16)
qry = torch.nn.functional.normalize(torch.randn(Q, D, device=dev, generator=g), dim=1)
lo, hi = shard_bounds(N, world, rank)
ix = FlatIPDeviceIndex(D, storage="bf16", device=dev, row_offset=lo); ix.add_bf16_rows(cat[lo:hi].clone())
sh = ShardedFlatIndex.from_device_index(ix, peer_exchange=os.environ.get("PEER", "1") == "1")
full = FlatIPDeviceIndex(D, storage="bf16", device=dev); full.add_bf16_rows(cat)
qo, qf = ix.prepare_queries(qry, normalize=False), full.prepare_queries(qry, normalize=False)
rng = np.random.default_rng(11)                                      # same seed on every rank: same global calls
live = np.ones(N, bool)
ok_all = True


def filters():
    out = {}
    for f in (0.9, 0.05):                                            # bitmap and compact shard paths
        rows = np.sort(rng.permutation(N)[: int(f * N)])
        out[f"filter f={f:g}"] = (sh.row_filter(rows=rows), full.row_filter(rows=rows))
    return out


def check(name, sels):
    global ok_all
    for k in (10, 100, 1000):
        s, i = sh.search(qo, k)
        s1, i1 = full.search_device(qf, k)
        ok = bool(torch.equal(i, i1) and torch.equal(s, s1))
        for fname, (sel, fsel) in sels.items():
            s, i = sh.search(qo, k, sel=sel)
            s1, i1 = full.search_device(qf, k, sel=fsel)
            ok &= bool(torch.equal(i, i1) and torch.equal(s, s1))
            if k == 100:
                h = sh.search_numpy(qry.cpu().numpy(), k, sel=sel)
                ok &= bool(np.array_equal(h[1], i1.cpu().numpy()) and np.array_equal(h[0], s1.cpu().numpy()))
        ok_all &= ok
        print(f"rank {rank}/{world} k={k} {name}: sharded == single: {ok}", flush=True)
    n = sh.n_live()
    ok_all &= n == full.n_live == int(live.sum())


def update(rows, normalize=True):
    x = rng.standard_normal((rows.size, D)).astype(np.float32)
    sh.update_rows(rows, x, normalize=normalize)
    full.update_rows(rows, x, normalize=normalize)
    live[rows] = True


def remove(rows):
    global ok_all
    mine = np.unique(rows)
    mine = mine[(mine >= ix.row_offset) & (mine < ix.row_offset + ix.ntotal)]
    n_here = int(live[mine].sum())
    ok_all &= sh.remove_rows(rows) == n_here
    full.remove_rows(rows)
    live[rows] = False


sels = filters()
check("unmutated", sels)
bounds = [shard_bounds(N, world, r)[0] for r in range(1, world)]
rows = rng.integers(0, N, size=20_000)
for j, b in enumerate(bounds):                                       # straddle every boundary, duplicates included
    rows[40 * j: 40 * j + 40] = np.concatenate([b - 10 + np.arange(20), b + 9 - np.arange(20)])
update(rows)
remove(rng.integers(0, N, size=N // 100))
check("updates + 1 % removed", sels)
llo, lhi = shard_bounds(N, world, world - 1)
remove(np.arange(llo + 500, lhi))
check("last shard keeps 500 rows", sels)
update(np.flatnonzero(~live)[::997][:1000])                          # freed slots take new items
check("revived", sels)
remap = sh.compact()
remap_full = full.compact()
ok_all &= bool(np.array_equal(remap, remap_full))
for sel, _ in sels.values():
    try:
        sh.search(qo, 100, sel=sel)
        ok_all = False
    except ValueError:
        pass
live = np.ones(full.ntotal, bool)
N = full.ntotal
print(f"rank {rank}/{world}: compacted to {N} rows, row_offset {ix.row_offset}, same map as the single index: "
      f"{bool(np.array_equal(remap, remap_full))}", flush=True)
check("compacted", filters())
remove(rng.integers(0, N, size=1000))
check("compacted, removed again", filters())
if rank == 0:
    print(f"peer exchange active: {any(k_[0] == 'peer' and v is not None for k_, v in sh._ids_cache.items())}")
flag = torch.tensor([1 if ok_all else 0], dtype=torch.int32, device=dev)
dist.all_reduce(flag, op=dist.ReduceOp.MIN)
dist.destroy_process_group()
sys.exit(0 if int(flag.item()) == 1 else 1)
