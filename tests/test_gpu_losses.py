"""The training losses against fp64, row by row and element by element: the in-batch forward on each of its four paths
(three stream_scores_kernel<NQ, BN, LseEpi> instantiations and the GEMM + lse_rows fallback), the six fused backward
instantiations and their work splits, the chunked backward, the explicit-negative loss and compute_similarity.  Every
in-batch case first asserts through the plan query (tests/loss_plan.py) that it reaches the path named in its id.

Two kinds of data:
- "exact": multiples of 1/8, so every logit is exact in fp32 under any piece count and only the fp32 exp / log / sums
  remain (about 1e-6 relative per row).  Users are +1/2 and items -1/2 per component, plus noise: every logit is
  strongly negative, so a padding row counted as a zero logit, a dropped partial or a misplaced tile moves lse by O(1).
- "random": normalised fp32 rows whose positives lean towards their user.  The logits carry the error of the piece
  products (see _eps_logit), which the tolerances follow.  In bf16 mode the reference is computed on bf16-rounded
  operands, whose products are exact in fp32."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from loss_plan import grad_plan, lse_path  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _exact(rows: int, E: int, sign: float, g: torch.Generator) -> torch.Tensor:
    return sign * (4 + torch.randint(-2, 3, (rows, E), generator=g)).float() / 8.0


def _random_pair(B: int, NI: int, E: int, diag0: int, g: torch.Generator, lean: float = 0.7):
    u = F.normalize(torch.randn(B, E, generator=g), dim=1)
    v = torch.randn(NI, E, generator=g)
    v[diag0:diag0 + B] = F.normalize(v[diag0:diag0 + B], dim=1) + lean * u
    return u, F.normalize(v, dim=1)


def _eps_logit(nprod: int, E: int, umax: float, vmax: float, inv_t: float) -> float:
    """Bound on the error of one logit <u, v> * inv_t computed from split-bf16 pieces with fp32 accumulation.
    1 product (bf16 mode, reference on the rounded operands): the products are exact, fp32 accumulation leaves at
    most E * 2^-24 of sum |u_k v_k| <= |u||v|.  3 products (h.h + m.h + h.m): bf16 rounds to 2^-8 relative, so
    x = h + m + r with |m| <= 2^-8 |x| and |r| <= 2^-16 |x|; the dropped m.m, r.(h + m), (h + m).r are
    <= 3 * 2^-16 |u_k v_k| < 2^-14 |u_k v_k|.  6 products: the dropped piece products are below the fp32 accumulation
    error."""
    rel = {1: E * 2.0 ** -23, 3: 2.0 ** -14 + E * 2.0 ** -23, 6: E * 2.0 ** -23}[nprod]
    return rel * umax * vmax * inv_t


def _norm_max(x: torch.Tensor) -> float:
    return float(x.double().norm(dim=1).max())


def _ref_lse(u: torch.Tensor, v: torch.Tensor, inv_t: float, chunk: int = 4096) -> torch.Tensor:
    """fp64 logsumexp_j(<u_b, v_j> * inv_t) per row, on the device in row chunks."""
    v64 = v.double()
    return torch.cat([torch.logsumexp(u[r0:r0 + chunk].double() @ v64.T * inv_t, 1) for r0 in range(0, u.shape[0], chunk)])


def _run_lse(u: torch.Tensor, v: torch.Tensor, terms: int, inv_t: float, path: str) -> torch.Tensor:
    """The forward's per-row lse on `path`: the fused kernel, or the fallback that ops.InBatchCEFn.forward runs."""
    from b200rec import kernels as K, ops
    B, NI = u.shape[0], v.shape[0]
    uo, vo = K.split_bf16(u, terms, 0), K.split_bf16(v, terms, 1)
    assert lse_path(B, NI, uo.stride(0)) == path
    lse = K.inbatch_lse(uo, vo, B, NI, inv_t)
    if path != "fallback":
        return lse
    assert lse is None
    parts = []
    for r0 in range(0, B, ops.InBatchCEFn.CHUNK):
        r1 = min(B, r0 + ops.InBatchCEFn.CHUNK)
        parts.append(K.lse_rows(K.gemm_tn(uo[r0:r1], vo, r1 - r0, NI, uo.shape[1]), inv_t, 0, False)[0])
    return torch.cat(parts)


# ------------------------------------------------------------------------------------------ in-batch forward, per row
# (path, B, NI, E, terms); terms = split-bf16 pieces of the operands: 1 in bf16 mode, 3 by default in fp32 mode,
# 6 with B200REC_LSE_TERMS=6 (tests/test_loss_plan_host.py pins the map)
LSE_CASES = [
    ("nq2bn128", 129, 129, 64, 3),
    ("nq2bn128", 255, 1000, 50, 3),
    ("nq2bn128", 257, 777, 128, 1),
    ("nq2bn128", 2049, 2086, 64, 3),
    ("nq2bn128", 8192, 8192, 64, 3),        # config 2 on one GPU
    ("nq1bn256", 1, 1, 64, 3),
    ("nq1bn256", 2, 65_573, 64, 3),         # one supertile in 129 partials
    ("nq1bn256", 127, 300, 32, 6),
    ("nq1bn256", 128, 128, 100, 3),
    ("nq1bn256", 1000, 1037, 128, 3),       # config 4 / ML-1M width, B > 128: BN = 256 still
    ("nq1bn64", 2, 65_573, 128, 6),         # one supertile in 148 partials
    ("nq1bn64", 129, 1000, 192, 3),
    ("nq1bn64", 257, 300, 100, 6),
    ("nq1bn64", 1, 70, 256, 3),
    ("fallback", 1, 70, 320, 3),
    ("fallback", 257, 1000, 192, 6),
    ("fallback", 2049, 2112, 320, 3),       # crosses the fallback's 2048-row chunk
    ("fallback", 127, 4133, 256, 6),
]


@pytest.mark.parametrize("kind", ["exact", "random"])
@pytest.mark.parametrize("path,B,NI,E,terms", LSE_CASES,
                         ids=[f"{c[0]}-B{c[1]}-NI{c[2]}-E{c[3]}-t{c[4]}" for c in LSE_CASES])
def test_inbatch_lse_per_row_matches_fp64(path, B, NI, E, terms, kind):
    g = torch.Generator().manual_seed(B * 7 + NI + E + terms)
    if kind == "exact":
        u, v, inv_t = _exact(B, E, 1.0, g), _exact(NI, E, -1.0, g), 1.0
    else:
        u, v = _random_pair(B, NI, E, 0, g, lean=0.5)
        inv_t = 20.0
    u, v = u.to(DEV), v.to(DEV)
    lse = _run_lse(u, v, terms, inv_t, path).double()
    ru, rv = (u.bfloat16().float(), v.bfloat16().float()) if terms == 1 else (u, v)
    ref = _ref_lse(ru, rv, inv_t)
    # fp32 exp2 / log2 and the sums over up to 65k terms, in sequence across tiles and partials: 1e-5 relative
    tol = 1e-5 * (1 + ref.abs())
    if kind == "random":
        # lse is a softmax-weighted mean of the logits, so it carries at most the bound of one logit
        tol = tol + _eps_logit(terms, E, _norm_max(ru), _norm_max(rv), inv_t)
    err = (lse - ref).abs()
    assert torch.isfinite(lse).all()
    assert (err <= tol).all(), (f"{int((err > tol).sum())} rows off, worst row {int((err / tol).argmax())}: "
                                f"err {float(err.max()):.3g}")


# (B, NI, diag0, total_rows, temperature, E, norm): diag0 = 0, a middle rank, the last rank (NI - B)
CE_CASES = [
    (1000, 1000, 0, 1000, 0.05, 64, 1.0),
    (512, 2085, 1024, 2048, 1.0, 128, 1.0),
    (300, 2100, 1800, 2100, 0.05, 64, 1.0),
    (700, 700, 0, 700, 0.02, 64, 5.0),        # norms up to 5 at T = 0.02: logits in the thousands
    (257, 900, 643, 1800, 0.02, 128, 5.0),
    (257, 600, 343, 600, 0.05, 320, 5.0),     # the fallback forward
]


@pytest.mark.parametrize("B,NI,diag0,total,T,E,norm", CE_CASES,
                         ids=[f"B{c[0]}-NI{c[1]}-diag{c[2]}-rows{c[3]}-T{c[4]}-E{c[5]}-norm{c[6]}" for c in CE_CASES])
def test_inbatch_ce_forward_with_offset_matches_fp64(B, NI, diag0, total, T, E, norm):
    """ops.InBatchCEFn forward in fp32 mode (3-term logits): sum_b(lse_b - <u_b, v_{diag0+b}>/T) / total_rows."""
    from b200rec import ops
    g = torch.Generator().manual_seed(B + NI + diag0)
    u, v = _random_pair(B, NI, E, diag0, g)
    if norm != 1.0:   # row norms spread over [0.2, norm]
        u = u * (0.2 + (norm - 0.2) * torch.rand(B, 1, generator=g))
        v = v * (0.2 + (norm - 0.2) * torch.rand(NI, 1, generator=g))
    u, v = u.to(DEV), v.to(DEV)
    inv_t = 1.0 / T
    assert lse_path(B, NI, 3 * ((E + 63) // 64 * 64)) == ("fallback" if E == 320 else ("nq2bn128" if E == 64 else "nq1bn256"))
    loss = ops.InBatchCEFn.apply(u, v, inv_t, 6, diag0, total).item()
    lse = _ref_lse(u, v, inv_t)
    pos = (u.double() * v[diag0:diag0 + B].double()).sum(1) * inv_t
    ref = float((lse - pos).sum() / total)
    # per row: the logit bound (3 products) on lse, fp32 rounding of lse and of pos (a row dot of E terms)
    eps = _eps_logit(3, E, _norm_max(u), _norm_max(v), inv_t)
    norms = u.double().norm(dim=1) * v[diag0:diag0 + B].double().norm(dim=1) * inv_t
    tol_rows = eps + 1e-5 * (1 + lse.abs() + pos.abs()) + E * 2.0 ** -23 * norms
    assert abs(loss - ref) <= float(tol_rows.sum()) / total, (loss, ref)


# ------------------------------------------------------------------------------------------------ in-batch backward
def _ref_grads(u, v, inv_t, diag0, coef, eps_logit, c_g):
    """fp64 dU, dV of sum_b(lse_b - s_{b, diag0+b}) * coef / inv_t, i.e. G = coef * (softmax - onehot), and element-wise
    error bounds for a kernel that evaluates G with logits off by up to eps_logit (lse too), rounds G and the other
    side's operand to c_g relative, and accumulates in fp32 (2^-13 of the absolute sum covers truncating tensor-core
    adds along chains of up to 400 partial products, split-K atomics and the final adds)."""
    B = u.shape[0]
    u64, v64 = u.double(), v.double()
    S = u64 @ v64.T * inv_t
    P = torch.exp(S - torch.logsumexp(S, 1, keepdim=True))
    ar = torch.arange(B, device=u.device)
    G = P.clone()
    G[ar, diag0 + ar] -= 1.0
    G *= coef
    W = (c_g + 2.0 ** -13) * G.abs() + 2.0 * eps_logit * coef * P
    return G @ v64, G.T @ u64, W @ v64.abs(), W.T @ u64.abs()


def _assert_within(name, got, ref, bound):
    err = (got.double() - ref).abs()
    ok = err <= bound + 1e-30
    assert torch.isfinite(got).all(), f"{name}: non-finite values"
    assert ok.all(), (f"{name}: {int((~ok).sum())} of {ok.numel()} elements outside the bound, first at "
                      f"{tuple(int(i) for i in (~ok).nonzero()[0])}, worst err/bound {float((err / (bound + 1e-30)).max()):.3g}")


# (E, operand terms, nprod_s, nprod_g, B, NI, diag0, split): operand terms 1 = bf16 mode, 3 = fp32 mode,
# 6 = B200REC_BWD_TERMS=6 (6-product recompute) or B200REC_LSE_TERMS=6 (3 products read from the 6-term layout)
FUSED_CASES = [
    (64, 1, 1, 1, 1000, 1000, 0, "none"),
    (128, 1, 1, 1, 1000, 1020, 20, "none"),    # 16 column tiles on both sides: one unit per row tile
    (64, 3, 3, 3, 2049, 2049, 0, "none"),
    (128, 3, 3, 3, 777, 2000, 1223, "u"),      # any NI with more 64-row tiles than B splits the user side
    (64, 6, 6, 3, 1000, 1000, 0, "none"),
    (128, 6, 6, 3, 513, 1500, 700, "u"),
    (64, 6, 3, 3, 1000, 1000, 0, "none"),
    (128, 6, 3, 3, 700, 1000, 300, "u"),
    (64, 3, 3, 3, 1024, 4133, 3109, "u"),
    (128, 1, 1, 1, 300, 9000, 4000, "u"),
    (64, 3, 3, 3, 8256, 8256, 0, "uv"),
    (128, 1, 1, 1, 8193, 8193, 0, "uv"),
    (128, 6, 6, 3, 8193, 8693, 500, "uv"),
]


@pytest.mark.parametrize("E,terms,nps,npg,B,NI,diag0,split", FUSED_CASES,
                         ids=[f"E{c[0]}-t{c[1]}-p{c[2]}{c[3]}-B{c[4]}-NI{c[5]}-diag{c[6]}-atomic_{c[7]}" for c in FUSED_CASES])
def test_fused_inbatch_backward_matches_fp64(E, terms, nps, npg, B, NI, diag0, split):
    """inbatch_grad_kernel<E, nps, npg> called directly with the fp64 lse, an upstream gradient of 2.5 through coef_dev
    and total_rows = NI; both outputs start as NaN, so a row the kernel leaves unwritten or adds into unzeroed shows."""
    from b200rec import kernels as K
    plan = grad_plan(B, NI, E, nps, npg)
    assert plan["supported"] == 1
    assert (plan["atomic_u"], plan["atomic_v"]) == (int("u" in split), int("v" in split)), plan
    g = torch.Generator().manual_seed(E + B + NI + nps)
    u, v = _random_pair(B, NI, E, diag0, g)
    u, v = u.to(DEV), v.to(DEV)
    inv_t, total, upstream = 20.0, NI, 2.5
    ru, rv = (u.bfloat16().float(), v.bfloat16().float()) if terms == 1 else (u, v)
    lse = _ref_lse(ru, rv, inv_t).float()
    uo, vo = K.split_bf16(u, terms, 0), K.split_bf16(v, terms, 1)
    dU = torch.full_like(u, float("nan"))
    dV = torch.full_like(v, float("nan"))
    K.inbatch_grad(uo, K.PIECE_BLOCKS[(terms, 0)], vo, K.PIECE_BLOCKS[(terms, 1)], B, NI, E, nps, npg, inv_t, lse,
                   diag0, inv_t / total, torch.tensor([upstream], device=DEV), dU, dV)
    # lse was rounded to fp32: 2^-24 |lse| on every exponent, below the logit bound
    eps = _eps_logit(nps, E, _norm_max(ru), _norm_max(rv), inv_t) + 2.0 ** -23 * float(lse.abs().max())
    c_g = 2.0 ** -8 if npg == 1 else 2.0 ** -14     # G rounded to bf16, or h + m pieces with 3 products
    rdU, rdV, bU, bV = _ref_grads(ru, rv, inv_t, diag0, upstream * inv_t / total, eps, c_g)
    _assert_within("dU", dU, rdU, bU)
    _assert_within("dV", dV, rdV, bV)


# (E, model terms, B, NI, diag0, env): the backward that ops.InBatchCEFn runs, end to end
E2E_CASES = [
    (32, 6, 2048, 2048, 0, {}),
    (100, 6, 2049, 2086, 37, {}),
    (192, 6, 4097, 4097, 0, {}),
    (100, 1, 2049, 2049, 0, {}),
    (64, 1, 2049, 4098, 2049, {"B200REC_INBATCH_BWD": "chunked"}),
    (128, 6, 2048, 2048, 0, {"B200REC_INBATCH_BWD": "chunked"}),
    (64, 6, 1000, 1000, 0, {"B200REC_LSE_TERMS": "6"}),
    (128, 6, 700, 1400, 700, {"B200REC_LSE_TERMS": "6"}),
]


@pytest.mark.parametrize("E,terms,B,NI,diag0,env", E2E_CASES,
                         ids=[f"E{c[0]}-t{c[1]}-B{c[2]}-NI{c[3]}-diag{c[4]}-" + ("-".join(f"{k[8:]}={v}" for k, v in c[5].items()) or "default")
                              for c in E2E_CASES])
def test_inbatch_ce_backward_paths_match_fp64(E, terms, B, NI, diag0, env, monkeypatch):
    """The chunked backward (E outside the fused instantiations, or B200REC_INBATCH_BWD=chunked) across its 2048-row
    chunks, and the fused one fed from 6-term operands (B200REC_LSE_TERMS=6, 3-product recompute)."""
    from b200rec import ops
    for k, val in env.items():
        monkeypatch.setenv(k, val)
    lse_terms = ops._lse_terms(terms)
    nps = 1 if terms == 1 else 3
    fused = env.get("B200REC_INBATCH_BWD") != "chunked" and grad_plan(B, NI, E, nps, nps)["supported"] == 1
    assert fused == ("B200REC_LSE_TERMS" in env)
    assert lse_terms == (6 if "B200REC_LSE_TERMS" in env else (1 if terms == 1 else 3))
    g = torch.Generator().manual_seed(E + B + terms)
    u, v = _random_pair(B, NI, E, diag0, g)
    uc, vc = u.to(DEV).requires_grad_(), v.to(DEV).requires_grad_()
    inv_t, upstream = 20.0, 2.5
    loss = ops.InBatchCEFn.apply(uc, vc, inv_t, terms, diag0, NI)
    (loss * upstream).backward()
    ru, rv = (u.bfloat16().float(), v.bfloat16().float()) if terms == 1 else (u, v)
    ru, rv = ru.to(DEV), rv.to(DEV)
    # the forward's lse carries the logit bound of lse_terms products; the recomputed logits that of lse_terms
    # (chunked) or of 3 products (fused, fp32 mode); _ref_grads doubles the sum for good measure
    eps = _eps_logit(lse_terms, E, _norm_max(ru), _norm_max(rv), inv_t) + _eps_logit(nps, E, _norm_max(ru), _norm_max(rv), inv_t)
    c_g = 2.0 ** -8 if terms == 1 else 2.0 ** -14
    rdU, rdV, bU, bV = _ref_grads(ru, rv, inv_t, diag0, upstream * inv_t / NI, eps, c_g)
    _assert_within("dU", uc.grad, rdU, bU)
    _assert_within("dV", vc.grad, rdV, bV)


# ------------------------------------------------------------------------------------------------ explicit negatives
def _ref_explicit(u, p, n, R, inv_t, bias_sum):
    """fp64 restatement of oracle.two_tower.explicit_loss per row: logits [<u,p>/T + biases | <u,n_j>/T], label 0."""
    B, E = u.shape
    u64, p64, n64 = u.double(), p.double(), n.double().reshape(B, R, E)
    logits = torch.cat([((u64 * p64).sum(1) * inv_t + bias_sum)[:, None], torch.einsum("be,bre->br", u64, n64) * inv_t], 1)
    lse = torch.logsumexp(logits, 1)
    P = torch.exp(logits - lse[:, None])
    dl = P.clone()
    dl[:, 0] -= 1.0
    du = (dl[:, :1] * p64 + torch.einsum("br,bre->be", dl[:, 1:], n64)) * inv_t
    dp = dl[:, :1] * u64 * inv_t
    dn = (dl[:, 1:, None] * u64[:, None, :] * inv_t).reshape(B * R, E)
    return lse - logits[:, 0], du, dp, dn, dl[:, 0], logits, P, dl


EXPLICIT_CASES = [(1, 1, 1), (7, 2, 7), (7, 31, 33), (7, 32, 64), (7, 33, 128), (7, 1535, 33), (7, 1536, 64),
                  (1, 2048, 300), (7, 4095, 128), (20_000, 2, 33), (20_000, 16, 64), (20_000, 33, 7)]


@pytest.mark.parametrize("bias", [False, True], ids=["nobias", "bias"])
@pytest.mark.parametrize("B,R,E", EXPLICIT_CASES, ids=[f"B{c[0]}-R{c[1]}-E{c[2]}" for c in EXPLICIT_CASES])
def test_explicit_ce_per_row_matches_fp64(B, R, E, bias):
    """b200rec_explicit_ce row losses and gradients (R >= 1536 needs more than 48 KB of shared memory per block; B =
    20,000 is beyond warp_rows_grid's 148 x 16 blocks of 8 rows, so warps loop over rows), then ops.ExplicitCEFn's mean
    and autograd with an upstream gradient of 2.5."""
    from b200rec import kernels as K, ops
    g = torch.Generator().manual_seed(B + R + E)
    u = F.normalize(torch.randn(B, E, generator=g), dim=1)
    p = F.normalize(torch.randn(B, E, generator=g) + 0.5 * u, dim=1)
    n = F.normalize(torch.randn(B * R, E, generator=g), dim=1)
    u, p, n = u.to(DEV), p.to(DEV), n.to(DEV)
    ub = torch.tensor([0.3], device=DEV) if bias else None
    ib = torch.tensor([-0.1], device=DEV) if bias else None
    bias_sum = 0.2 if bias else 0.0
    inv_t, gs = 20.0, 0.75
    row, du, dp, dn, dbias = K.explicit_ce(u, p, n, R, inv_t, ub, ib, grad_scale=gs,
                                           grad_scale_dev=torch.tensor([2.0], device=DEV), want_grad=True)
    rrow, rdu, rdp, rdn, rdb, logits, P, dl = _ref_explicit(u, p, n, R, inv_t, float(np.float32(0.3) + np.float32(-0.1)) if bias else 0.0)
    # logits are fp32 dot products of unit rows (E * 2^-24 * inv_t) scaled in fp32; lse and the difference in fp32
    eps = E * 2.0 ** -23 * inv_t + 2.0 ** -22 * float(logits.abs().max())
    _assert_within("row_loss", row, rrow, 2 * eps + 1e-6 * (1 + logits.abs().max(1).values))
    # gradients: dlogit_j = p_j - [j == 0] with p_j off by p_j * 2 eps and fp32 rounding, times the scale 0.75 * 2.0;
    # dU sums R + 1 terms in sequence in fp32: (R + 2) * 2^-24 of the absolute sum
    scale = gs * 2.0
    w = (2.0 * eps * P + 2.0 ** -20 * (dl.abs() + P)) * scale        # [B, R+1] bound on each scaled dlogit
    n3a = n.double().abs().reshape(B, R, E)
    bu = (w[:, :1] * p.double().abs() + torch.einsum("br,bre->be", w[:, 1:], n3a)) * inv_t + ((R + 2) * 2.0 ** -24) * (
        (dl.abs()[:, :1] * p.double().abs() + torch.einsum("br,bre->be", dl.abs()[:, 1:], n3a)) * inv_t * scale)
    _assert_within("dU", du, rdu * scale, bu)
    _assert_within("dP", dp, rdp * scale, (w[:, :1] + 2.0 ** -22 * scale) * u.double().abs() * inv_t)
    _assert_within("dN", dn, rdn * scale, ((w[:, 1:, None] + 2.0 ** -22 * scale) * u.double().abs()[:, None, :] * inv_t).reshape(B * R, E))
    _assert_within("row_dbias", dbias, rdb * scale, w[:, 0])
    # mean loss and autograd (grad_scale = upstream / B from the device)
    uc, pc, nc = (t.clone().requires_grad_() for t in (u, p, n))
    ubc = ub.clone().requires_grad_() if bias else None
    ibc = ib.clone().requires_grad_() if bias else None
    loss = ops.ExplicitCEFn.apply(uc, pc, nc, ubc, ibc, inv_t)
    assert abs(loss.item() - float(rrow.mean())) <= float(2 * eps + 1e-6 * (1 + logits.abs().max()))
    (loss * 2.5).backward()
    s = 2.5 / B / scale
    _assert_within("autograd dU", uc.grad, rdu * 2.5 / B, bu * s)
    _assert_within("autograd dP", pc.grad, rdp * 2.5 / B, (w[:, :1] * s + 2.0 ** -22 * 2.5 / B) * u.double().abs() * inv_t)
    if bias:
        want = float(rdb.sum()) * 2.5 / B
        for b in (ubc, ibc):
            assert abs(b.grad.item() - want) <= float(w[:, 0].sum()) * s + 1e-6 * abs(want)


def test_explicit_ce_fp64_restatement_matches_the_oracle():
    """The torch restatement above against oracle.two_tower.explicit_loss (numpy) on a small shape with biases."""
    from oracle.two_tower import explicit_loss
    rng = np.random.default_rng(3)
    B, R, E, T = 5, 37, 33, 0.05
    u, p, n = (rng.standard_normal(s) for s in ((B, E), (B, E), (B * R, E)))
    loss, du, dp, dn, db = explicit_loss(u, p, n, T, 0.3, -0.1, want_grad=True)
    rrow, rdu, rdp, rdn, rdb, *_ = _ref_explicit(*(torch.from_numpy(x) for x in (u, p, n)), R, 1 / T, 0.2)
    assert abs(float(rrow.mean()) - loss) <= 1e-12 * max(1.0, abs(loss))
    for got, want in ((rdu / B, du), (rdp / B, dp), (rdn / B, dn)):
        np.testing.assert_allclose(got.numpy(), want, rtol=1e-10, atol=1e-14)
    assert abs(float(rdb.sum()) / B - db) <= 1e-12


# ------------------------------------------------------------------------------------------------ compute_similarity
@pytest.mark.parametrize("bias", [False, True], ids=["nobias", "bias"])
@pytest.mark.parametrize("B,E", [(1, 1), (1, 128), (20_000, 33), (40_000, 1), (40_000, 128)])
def test_compute_similarity_matches_fp64(B, E, bias):
    """ops.RowDotFn: rowdot_kernel (grid-stride beyond 18,944 rows), rowdot_bwd_kernel (grid-stride beyond 606,208
    elements) and the bias gradient through ce_sum (fp64 sum in one block)."""
    from b200rec import ops
    g = torch.Generator().manual_seed(B + E)
    u, i = torch.randn(B, E, generator=g).to(DEV), torch.randn(B, E, generator=g).to(DEV)
    up = torch.randn(B, generator=g).to(DEV)
    ub = torch.tensor([0.3], device=DEV, requires_grad=True) if bias else None
    ib = torch.tensor([-0.7], device=DEV, requires_grad=True) if bias else None
    uc, ic = u.clone().requires_grad_(), i.clone().requires_grad_()
    inv_t = 20.0
    out = ops.RowDotFn.apply(uc, ic, ub, ib, inv_t)
    (out * up).sum().backward()
    dots = (u.double() * i.double()).sum(1)
    ref = dots * inv_t + (float(np.float32(0.3) + np.float32(-0.7)) if bias else 0.0)
    absdot = (u.double().abs() * i.double().abs()).sum(1)
    _assert_within("similarity", out, ref, (E * 2.0 ** -23 * absdot + 2.0 ** -23 * dots.abs()) * inv_t + 2.0 ** -22 * ref.abs() + 1e-7)
    _assert_within("dU", uc.grad, up.double()[:, None] * inv_t * i.double(), 2.0 ** -22 * (up.double().abs()[:, None] * inv_t * i.double().abs()))
    _assert_within("dI", ic.grad, up.double()[:, None] * inv_t * u.double(), 2.0 ** -22 * (up.double().abs()[:, None] * inv_t * u.double().abs()))
    if bias:
        want = float(up.double().sum())
        for b in (ub, ib):
            assert abs(b.grad.item() - want) <= 2.0 ** -22 * float(up.double().abs().sum()) + 1e-6 * abs(want)
