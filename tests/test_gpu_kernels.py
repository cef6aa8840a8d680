"""GPU parity tests of the low-level kernels, called through the C-ABI (ctypes) and checked against the CPU oracle."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

pytestmark = pytest.mark.gpu


def _bf16_round(x: torch.Tensor) -> torch.Tensor:
    return x.to(torch.bfloat16).to(torch.float32)


@pytest.mark.parametrize("M,N,K", [(128, 128, 64), (100, 17, 20), (1024, 256, 3), (300, 128, 256), (4096, 64, 128)])
@pytest.mark.parametrize("terms", [1, 6])
def test_gemm_matches_fp32(M, N, K, terms):
    from b200rec import kernels as KR
    g = torch.Generator().manual_seed(M * 7 + N * 3 + K)
    x = torch.randn(M, K, generator=g)
    w = torch.randn(N, K, generator=g) / K ** 0.5
    b = torch.randn(N, generator=g)
    out = KR.matmul_nt(x.cuda(), w.cuda(), b.cuda(), terms=terms).cpu()
    if terms == 1:
        ref = _bf16_round(x).double() @ _bf16_round(w).double().T + b.double()
        tol = 1e-5
    else:
        ref = x.double() @ w.double().T + b.double()
        tol = 5e-6
    err = (out.double() - ref).abs().max().item()
    scale = ref.abs().max().item()
    assert err <= tol * max(scale, 1.0), f"gemm {M}x{N}x{K} terms={terms}: max abs err {err:.3e} (scale {scale:.3e})"


def test_gemm_split_k():
    from b200rec import kernels as KR
    g = torch.Generator().manual_seed(5)
    x = torch.randn(96, 5000, generator=g)
    w = torch.randn(40, 5000, generator=g)
    xo, wo = KR.split_bf16(x.cuda(), 6, 0), KR.split_bf16(w.cuda(), 6, 1)
    out = KR.gemm_tn(xo, wo, 96, 40, xo.shape[1], None, 0.5, k_splits=16).cpu()
    ref = 0.5 * (x.double() @ w.double().T)
    assert (out.double() - ref).abs().max().item() <= 2e-4


def test_split_transpose():
    from b200rec import kernels as KR
    g = torch.Generator().manual_seed(6)
    x = torch.randn(70, 130, generator=g)
    w = torch.randn(50, 130, generator=g)
    # x^T [130,70] . w^T[130,50]^T  = x^T w  -> [70... ] check  (x^T)(w^T)^T = x^T w  is [130? no]
    a = KR.split_bf16(x.cuda(), 6, 0, transpose=True)   # [130, 6*128]
    b = KR.split_bf16(w.cuda(), 6, 1, transpose=True)   # [130, 6*64]
    assert a.shape == (130, 6 * 128) and b.shape == (130, 6 * 64)
    # contraction needs equal K: use x^T [130,70] against y^T with y [33,70]... build directly
    y = torch.randn(33, 70, generator=g)
    yo = KR.split_bf16(y.cuda(), 6, 1)                   # [33, 6*128]
    out = KR.gemm_tn(a, yo, 130, 33, a.shape[1]).cpu()   # x^T y^T = (y x)^T
    ref = (x.double().T @ y.double().T)
    assert (out.double() - ref).abs().max().item() <= 2e-5


def _oracle_topk(cat, qry, k, exclude=None):
    from oracle.flat_ip import IndexFlatIP
    ix = IndexFlatIP(cat.shape[1])
    ix.add(cat)
    return ix.search(qry, k, exclude=exclude)


def _check_topk(D, I, rD, rI, cat, qry):
    D, I = D.cpu().numpy(), I.cpu().numpy()
    # scores: tensor-core fp32 accumulation of exact bf16 products vs numpy sgemm
    assert np.allclose(D, rD, atol=2e-5, rtol=0), f"scores differ: max {np.abs(D - rD).max():.3e}"
    same = I == rI
    if not same.all():
        # ids may legitimately differ only inside groups of scores tied within 1e-5 (north_star tolerance)
        bad = np.argwhere(~same)
        for qi, j in bad[:2000]:
            s_ref = rD[qi, j]
            s_got = float(cat[I[qi, j]].astype(np.float64) @ qry[qi].astype(np.float64)) if I[qi, j] >= 0 else None
            assert s_got is not None and abs(s_got - s_ref) <= 1e-5, \
                f"query {qi} rank {j}: got id {I[qi, j]} (score {s_got}) want {rI[qi, j]} (score {s_ref})"
    for qi in range(D.shape[0]):
        valid = I[qi] >= 0
        assert len(set(I[qi][valid].tolist())) == valid.sum(), "duplicate ids in result"
        assert (np.diff(D[qi]) <= 0).all(), "scores not descending"


@pytest.mark.parametrize("N,Q,D,k", [(5000, 10, 128, 100), (20000, 130, 64, 10), (100000, 300, 128, 100),
                                     (70000, 600, 128, 100), (3000, 5, 192, 1000), (50, 3, 64, 100),
                                     (200000, 1100, 64, 37)])
def test_flat_ip_topk_matches_oracle(N, Q, D, k):
    from b200rec import kernels as KR
    from oracle.flat_ip import bf16_round, normalize_L2
    rng = np.random.default_rng(N + Q + D + k)
    cat = bf16_round(normalize_L2(rng.standard_normal((N, D)).astype(np.float32)))
    qry = bf16_round(normalize_L2(rng.standard_normal((Q, D)).astype(np.float32)))
    rD, rI = _oracle_topk(cat, qry, k)
    ld = (D + 63) // 64 * 64
    c = torch.zeros((N, ld), dtype=torch.bfloat16, device="cuda")
    q = torch.zeros((Q, ld), dtype=torch.bfloat16, device="cuda")
    c[:, :D] = torch.from_numpy(cat).cuda().to(torch.bfloat16)
    q[:, :D] = torch.from_numpy(qry).cuda().to(torch.bfloat16)
    Dg, Ig = KR.flat_ip_topk(c, q, k)
    torch.cuda.synchronize()
    _check_topk(Dg, Ig, rD, rI, cat, qry)


def test_flat_ip_topk_ties_and_exclusion():
    from b200rec import kernels as KR
    rng = np.random.default_rng(3)
    N, Q, D, k = 40000, 140, 64, 50
    base = rng.integers(-2, 3, size=(N, D)).astype(np.float32)   # small integers: exact scores, massive ties
    qry = rng.integers(-2, 3, size=(Q, D)).astype(np.float32)
    excl = [np.sort(rng.choice(N, size=rng.integers(0, 300), replace=False)).astype(np.int32) for _ in range(Q)]
    rD, rI = _oracle_topk(base, qry, k, exclude=excl)
    c = torch.from_numpy(base).cuda().to(torch.bfloat16)
    q = torch.from_numpy(qry).cuda().to(torch.bfloat16)
    indptr = torch.tensor(np.concatenate([[0], np.cumsum([len(e) for e in excl])]), dtype=torch.int64, device="cuda")
    rows = torch.from_numpy(np.concatenate(excl)).cuda()
    Dg, Ig = KR.flat_ip_topk(c, q, k, exclude_indptr=indptr, exclude_rows=rows)
    torch.cuda.synchronize()
    # exact integer scores: the total order (score desc, row asc) must be reproduced bit for bit
    assert np.array_equal(Dg.cpu().numpy(), rD)
    assert np.array_equal(Ig.cpu().numpy(), rI)


@pytest.mark.parametrize("sched", ["default", "0", "3", "4"])
@pytest.mark.parametrize("N,Q,D,k", [(300_000, 1500, 64, 20), (150_000, 4500, 64, 10)])
def test_flat_ip_topk_work_splits_bit_exact(sched, N, Q, D, k):
    """The 2-CTA kernel's work decompositions (time-aligned strided sweep with idle leftover units, the same with
    leftover units that change supertile and hand their lists over, contiguous split) on integer data: exact scores,
    massive ties, so the total order (score desc, row asc) must come out bit for bit.  B200REC_SCHED is applied with
    b200rec_debug_reload_env() and the plan query proves which decomposition ran; sched=4 idles leftover units even on
    long scans, which on these shapes is the default decomposition (tests/test_topk_plan_host.py pins the long scan)."""
    from b200rec import kernels as KR
    from topk_plan import decomposition, plan, topk_knobs
    rng = np.random.default_rng(N + Q)
    base = rng.integers(-3, 4, size=(N, D)).astype(np.float32)
    qry = rng.integers(-3, 4, size=(Q, D)).astype(np.float32)
    rD, rI = _oracle_topk(base, qry, k)
    with topk_knobs(B200REC_SCHED=None if sched == "default" else sched):
        p = plan(N, D, Q, k)
        split = {"default": "aligned-idle", "0": "contiguous", "3": "aligned-working", "4": "aligned-idle"}[sched]
        assert p["v2"] == 2 and decomposition(p) == split, p
        Dg, Ig = KR.flat_ip_topk(torch.from_numpy(base).cuda().to(torch.bfloat16),
                                 torch.from_numpy(qry).cuda().to(torch.bfloat16), k)
        torch.cuda.synchronize()
    assert np.array_equal(Dg.cpu().numpy(), rD)
    assert np.array_equal(Ig.cpu().numpy(), rI)


def test_flat_ip_topk_more_supertiles_than_units():
    """Q so large that there are more 512-query supertiles than CTA pairs: contiguous split, units that cross several
    supertiles."""
    from b200rec import kernels as KR
    rng = np.random.default_rng(77)
    N, Q, D, k = 12_000, 38_500, 64, 10
    base = rng.integers(-3, 4, size=(N, D)).astype(np.float32)
    qry = rng.integers(-3, 4, size=(Q, D)).astype(np.float32)
    rD, rI = _oracle_topk(base, qry, k)
    Dg, Ig = KR.flat_ip_topk(torch.from_numpy(base).cuda().to(torch.bfloat16),
                             torch.from_numpy(qry).cuda().to(torch.bfloat16), k)
    torch.cuda.synchronize()
    assert np.array_equal(Dg.cpu().numpy(), rD)
    assert np.array_equal(Ig.cpu().numpy(), rI)


def test_flat_ip_topk_large_k_generic_merge():
    """k + list > 256 keys: the helper warps take the shared-memory histogram select instead of the register one."""
    from b200rec import kernels as KR
    from oracle.flat_ip import bf16_round, normalize_L2
    rng = np.random.default_rng(99)
    N, Q, D, k = 120_000, 300, 64, 300
    cat = bf16_round(normalize_L2(rng.standard_normal((N, D)).astype(np.float32)))
    qry = bf16_round(normalize_L2(rng.standard_normal((Q, D)).astype(np.float32)))
    rD, rI = _oracle_topk(cat, qry, k)
    Dg, Ig = KR.flat_ip_topk(torch.from_numpy(cat).cuda().to(torch.bfloat16),
                             torch.from_numpy(qry).cuda().to(torch.bfloat16), k)
    torch.cuda.synchronize()
    _check_topk(Dg, Ig, rD, rI, cat, qry)


def test_topk_merge_matches_oracle():
    from b200rec import kernels as KR
    from oracle.flat_ip import merge_topk
    rng = np.random.default_rng(11)
    parts, Q, kin, kout = 8, 77, 100, 100
    s = rng.standard_normal((parts, Q, kin)).astype(np.float32)
    s = np.round(s, 1)  # ties
    ids = np.stack([rng.permutation(100000)[: Q * kin].reshape(Q, kin) + p * 100000 for p in range(parts)]).astype(np.int64)
    ids[0, :, -5:] = -1
    rs, ri = merge_topk([s[p] for p in range(parts)], [ids[p] for p in range(parts)], kout)
    gs, gi = KR.topk_merge(torch.from_numpy(s).cuda(), torch.from_numpy(ids).cuda(), kout)
    assert np.array_equal(gs.cpu().numpy(), rs)
    assert np.array_equal(gi.cpu().numpy(), ri)


def test_sharded_search_with_shared_thresholds_single_gpu():
    """Two row shards emulated on one GPU: sample -> union k-th -> tau_init -> local top-K -> merge == oracle."""
    from b200rec import kernels as KR
    from b200rec.retrieval import FlatIPDeviceIndex
    from oracle.flat_ip import bf16_round, normalize_L2
    rng = np.random.default_rng(21)
    N, Q, D, k = 600_000, 300, 64, 50
    cat = bf16_round(normalize_L2(rng.standard_normal((N, D)).astype(np.float32)))
    qry = bf16_round(normalize_L2(rng.standard_normal((Q, D)).astype(np.float32)))
    rD, rI = _oracle_topk(cat, qry, k)
    shards = []
    for lo, hi in ((0, 250_000), (250_000, N)):
        ix = FlatIPDeviceIndex(D, storage="bf16", row_offset=lo)
        ix.add(cat[lo:hi])
        shards.append(ix)
    q_op = shards[0].prepare_queries(qry)
    assert all(ix.has_sample_pass(Q, k) for ix in shards)
    from b200rec.dist import ShardedFlatIndex
    kx = ShardedFlatIndex.exchange_width(k, 2)
    assert k // 2 < kx <= k
    vals = torch.stack([ix.sample_device(q_op, k, kx, 2) for ix in shards])     # [2, Q, kx]: thinned sample, kx maxima each
    ids = torch.arange(vals.numel(), device="cuda").view_as(vals)
    tau = KR.topk_merge(vals.contiguous(), ids.contiguous(), k)[0][:, k - 1].contiguous()
    assert torch.equal(tau, KR.topk_pooled_kth(vals.contiguous(), k))            # the one-launch form the shards use
    assert (tau.cpu().numpy() <= rD[:, k - 1] + 1e-6).all(), "shared threshold must be a lower bound of the k-th score"
    parts = [ix.search_device(q_op, k, tau_init=tau) for ix in shards]
    s = torch.stack([p[0] for p in parts]).contiguous()
    i = torch.stack([p[1] for p in parts]).contiguous()
    Dg, Ig = KR.topk_merge(s, i, k)
    torch.cuda.synchronize()
    _check_topk(Dg, Ig, rD, rI, cat, qry)
