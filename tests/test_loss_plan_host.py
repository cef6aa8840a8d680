"""CPU-side checks of the in-batch loss planners (no GPU): which forward log-sum-exp kernel and which fused backward
instantiation and work split each shape reaches, read back through the plan query `b200rec_debug_loss_plan`.
tests/test_gpu_losses.py runs these paths on the device and relies on what is pinned here."""
import ctypes as C
import os
import sys

import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from loss_plan import grad_plan, lse_path, pad64, plan  # noqa: E402

WIDTHS = (32, 50, 64, 100, 128, 192, 256, 320)
BATCHES = (1, 128, 129, 8192)


def _need_148_sms():
    if plan(8192, 8192, 192)["sms"] != 148:
        pytest.skip("the grid sizes are pinned for 148 SMs")


def _want_lse(B: int, ld: int) -> str:
    """The forward map, from the shared-memory budget of stream_scores_kernel (227 KB less barriers and the resident
    128 * NQ user rows, ld / 64 blocks of 16 KB per 128 rows): NQ = 2 needs 3 stages of 128 item rows, so ld <= 320,
    and is only taken for B > 128; BN = 256 needs 3 stages of 256 rows (ld <= 512); BN = 64 needs 2 stages of 64 rows
    (ld <= 832); wider operands go through the GEMM + lse_rows fallback."""
    if B > 128 and ld <= 320:
        return "nq2bn128"
    if ld <= 512:
        return "nq1bn256"
    if ld <= 832:
        return "nq1bn64"
    return "fallback"


@pytest.mark.parametrize("terms", [1, 3, 6])
def test_forward_map_cell_by_cell(terms):
    from b200rec import _native
    lib = _native.lib()
    seen = set()
    for E in WIDTHS:
        ld = terms * pad64(E)
        for B in BATCHES:
            for NI in (B, 4 * B + 37):   # the item count never changes the instantiation
                got = lse_path(B, NI, ld)
                assert got == _want_lse(B, ld), (terms, E, B, NI)
                # the workspace query is what ops.InBatchCEFn uses to choose the fallback: 0 exactly when there is no plan
                assert (lib.b200rec_inbatch_lse_workspace_bytes(B, NI, ld) == 0) == (got == "fallback")
                seen.add(got)
    # the model's widths reach every path: bf16 and 3 terms only the streaming kernels, 3 and 6 terms also the fallback
    assert seen == {1: {"nq1bn256", "nq2bn128"}, 3: {"nq1bn256", "nq2bn128", "nq1bn64", "fallback"},
                    6: {"nq1bn256", "nq1bn64", "fallback"}}[terms]


def test_forward_map_edges_and_partials():
    _need_148_sms()
    assert lse_path(129, 129, 320) == "nq2bn128" and lse_path(129, 129, 384) == "nq1bn256"
    assert lse_path(1, 1, 512) == "nq1bn256" and lse_path(1, 1, 576) == "nq1bn64"
    assert lse_path(1, 1, 832) == "nq1bn64" and lse_path(1, 1, 896) == "fallback"
    assert lse_path(1, 1, 100) == "fallback"            # not a multiple of 64: no streaming plan either
    # a few users against a large item batch: one supertile cut into many partials, merged by lse_merge_kernel
    p = plan(2, 65_536 + 37, 192)
    assert (p["lse_nq"], p["lse_bn"], p["lse_S"], p["lse_T"]) == (1, 256, 1, 257)
    assert p["lse_grid"] == 129 and p["lse_W"] == 2 and p["lse_max_parts"] == 129
    # the training shape of config 2 (B = 8192, E = 64, 3 terms): 32 supertiles of 256 users
    p = plan(8192, 8192, 192)
    assert (p["lse_nq"], p["lse_bn"], p["lse_S"], p["lse_T"], p["lse_grid"]) == (2, 128, 32, 64, 147)


@pytest.mark.parametrize("E", [64, 128])
@pytest.mark.parametrize("nps,npg", [(1, 1), (3, 3), (6, 3)])
def test_fused_backward_instantiations(E, nps, npg):
    from b200rec import kernels as K
    g = grad_plan(1000, 1000, E, nps, npg)
    assert g["supported"] == 1 and K.inbatch_grad_supported(1000, 1000, E, nps, npg)
    assert 2 <= g["NST"] <= 4 and g["smem"] <= 232448
    # (128, 6, 3) keeps 3 pieces of both operands resident: only 2 ring stages fit
    assert g["NST"] == (2 if (E, nps) == (128, 6) else 4)


@pytest.mark.parametrize("E,nps,npg", [(32, 3, 3), (100, 3, 3), (192, 1, 1), (256, 3, 3), (64, 3, 1), (64, 6, 6),
                                       (128, 1, 3), (64, 6, 1)])
def test_fused_backward_refuses_what_it_does_not_instantiate(E, nps, npg):
    from b200rec import kernels as K
    assert grad_plan(1000, 1000, E, nps, npg) == dict.fromkeys(grad_plan(1000, 1000, E, nps, npg), 0)
    assert not K.inbatch_grad_supported(1000, 1000, E, nps, npg)


@pytest.mark.parametrize("B,NI,split_u,split_v", [
    (8192, 8192, 1, 1),        # config 2 on one GPU: 128 column tiles of 64 per unit, no atomics
    (8193, 8193, 2, 2),        # one more row: 129 tiles on both sides, every row's columns split in two
    (8256, 8256, 2, 2),
    (2048, 2048, 1, 1),
    (1024, 4096, 4, 1),        # data parallel, 4 ranks: the item side's columns are the 1024 local users
    (8192, 65_536, 8, 1),      # data parallel, 8 ranks
    (8193, 16_386, 3, 2),
    (1, 1, 1, 1),
    (100, 7_000, 55, 1),      # 2 user tiles set the unit length: the 110 item tiles of a row take 55 units
])
def test_fused_backward_work_split(B, NI, split_u, split_v):
    """Units are a 128-row tile times at most 128 column tiles of 64 (IG_MAX_UNIT_TILES), and both sides use the same
    unit length: min(column tiles of U, of V, 128).  A side whose columns need more than one unit adds its partial rows
    with atomics into a zeroed output.  Since the positives lie inside the items (NI >= B), the V side never splits alone."""
    for E, nps, npg in ((64, 3, 3), (128, 1, 1)):
        g = grad_plan(B, NI, E, nps, npg)
        assert (g["splits_u"], g["splits_v"]) == (split_u, split_v), (E, g)
        assert (g["atomic_u"], g["atomic_v"]) == (int(split_u > 1), int(split_v > 1))
        assert g["units_u"] == (B + 127) // 128 * split_u


def test_plan_query_rejects_bad_arguments_without_a_launch():
    from b200rec import _native
    lib = _native.lib()
    before = lib.b200rec_launch_count()
    for B, NI in ((0, 10), (10, 0), (-1, 5)):
        with pytest.raises(RuntimeError, match="empty"):
            plan(B, NI, 192, 64, 3, 3)
    out = (C.c_longlong * 4)()
    assert lib.b200rec_debug_loss_plan(10, 10, 192, 64, 3, 3, None, 4) != 0
    assert "null" in _native.last_error()
    # a short output array receives the leading fields only
    assert lib.b200rec_debug_loss_plan(10, 10, 192, 64, 3, 3, out, 3) == 0
    assert list(out) == [plan(10, 10)["sms"], 1, 256, 0]
    assert lib.b200rec_launch_count() == before


def test_explicit_ce_refuses_more_than_4095_negatives_before_any_launch():
    """The kernel keeps R + 1 logits per warp in shared memory (128 KB at R = 4095, the largest it accepts)."""
    from b200rec import _native
    lib = _native.lib()
    before = lib.b200rec_launch_count()
    buf = (C.c_float * 16)()
    p = C.cast(buf, C.c_void_p)
    rc = lib.b200rec_explicit_ce(p, p, p, 1, 4096, 1, 1.0, None, None, p, 0.0, None, None, None, None, None, None)
    assert rc != 0 and "at most 4095" in _native.last_error()
    assert lib.b200rec_launch_count() == before
