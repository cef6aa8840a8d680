"""torchrun --nproc-per-node G tools/check_sharded_filtered.py : row-sharded FILTERED top-k == single-GPU filtered top-k on
the same rows, bit for bit, for random and skewed filters (PEER=1: peer-memory fan-out exchange, PEER=0: NCCL
all-gather).  Also checks the host pipeline (search_numpy(sel=)) and that the unfiltered search is unchanged.  Exits
non-zero on any mismatch."""
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
ix = FlatIPDeviceIndex(D, storage="bf16", device=dev, row_offset=lo); ix.add_bf16_rows(cat[lo:hi].contiguous())
sh = ShardedFlatIndex.from_device_index(ix, peer_exchange=os.environ.get("PEER", "1") == "1")
full = FlatIPDeviceIndex(D, storage="bf16", device=dev); full.add_bf16_rows(cat)
qo, qf = ix.prepare_queries(qry, normalize=False), full.prepare_queries(qry, normalize=False)
rng = np.random.default_rng(11)                                      # same seed on every rank: same global filters
r0 = shard_bounds(N, world, 0)
filters = {f"random f={f:g}": np.sort(rng.permutation(N)[: int(f * N)]) for f in (0.9, 0.5, 0.05, 0.001)}
filters["skewed: all on shard 0"] = np.sort(r0[0] + rng.permutation(r0[1] - r0[0])[: (r0[1] - r0[0]) // 10])
filters["skewed: 95 % on the last shard"] = np.unique(np.concatenate([
    rng.integers(*shard_bounds(N, world, world - 1), size=N // 50), rng.integers(0, N, size=N // 1000)]))
filters["fewer than k rows"] = np.sort(rng.permutation(N)[:37])
filters["empty"] = np.zeros(0, np.int64)
ok_all = True
for k in (10, 100, 1000):
    s, i = sh.search(qo, k)
    s1, i1 = full.search_device(qf, k)
    ok = bool(torch.equal(i, i1) and torch.equal(s, s1))
    ok_all &= ok
    print(f"rank {rank}/{world} k={k} unfiltered: sharded == single: {ok}", flush=True)
    for name, rows in filters.items():
        s, i = sh.search(qo, k, sel=sh.row_filter(rows=rows))
        s1, i1 = full.search_device(qf, k, sel=full.row_filter(rows=rows))
        ok = bool(torch.equal(i, i1) and torch.equal(s, s1))
        if k == 100:
            h = sh.search_numpy(qry.cpu().numpy(), k, sel=sh.row_filter(rows=rows))
            ok &= bool(np.array_equal(h[1], i1.cpu().numpy()) and np.array_equal(h[0], s1.cpu().numpy()))
        ok_all &= ok
        print(f"rank {rank}/{world} k={k} {name}: sharded filtered == single filtered: {ok}", flush=True)
if rank == 0:
    print(f"peer exchange active: {any(k_[0] == 'peer' and v is not None for k_, v in sh._ids_cache.items() if isinstance(k_, tuple))}")
flag = torch.tensor([1 if ok_all else 0], dtype=torch.int32, device=dev)
dist.all_reduce(flag, op=dist.ReduceOp.MIN)
dist.destroy_process_group()
sys.exit(0 if int(flag.item()) == 1 else 1)
