"""CPU-side checks of the exact top-K planner (no GPU): which kernel instantiation and work decomposition each shape and
development knob reaches, read back through the plan query `b200rec_debug_topk_plan`.  tests/test_gpu_topk_paths.py
runs these paths on the device and relies on what is pinned here."""
import os
import sys

import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from topk_plan import DEFAULT_MAP, KNOBS, decomposition, default_path, path_name, plan, topk_knobs  # noqa: E402

QS = (1, 128, 129, 256, 257, 513)


@pytest.fixture(autouse=True)
def _default_knobs(monkeypatch):
    """Every case starts from the default plans, whatever the calling environment sets."""
    for name in KNOBS:
        monkeypatch.delenv(name, raising=False)
    with topk_knobs():
        yield


def _need_148_sms():
    if plan(50_037, 64, 1, 10)["sms"] != 148:
        pytest.skip("the map is pinned for 148 SMs")


@pytest.mark.parametrize("ld", sorted(DEFAULT_MAP))
def test_default_map_cell_by_cell(ld):
    _need_148_sms()
    for q in QS:
        p = plan(50_037, ld, q, 10)
        assert path_name(p) == default_path(ld, q), (ld, q, p)
        assert p["ks"] == (1 if (ld // 64) % 2 or not p["v2"] else 2)


def test_default_map_ends_at_ld_768_with_a_message_and_no_launch():
    from b200rec import _native
    lib = _native.lib()
    before = lib.b200rec_launch_count()
    for ld in (768, 1024):
        with pytest.raises(RuntimeError, match="dimension too large"):
            plan(50_037, ld, 129, 10)
        assert lib.b200rec_topk_workspace_bytes(50_037, ld, 129, 10) == 0
        assert "dimension too large" in _native.last_error()
    assert lib.b200rec_topk_workspace_bytes(50_037, 704, 129, 10) > 0
    assert lib.b200rec_launch_count() == before


def test_plan_query_reports_the_flush_rule_and_list_capacity():
    _need_148_sms()
    # k > 128 with Q <= 256: lists are handed over only when full; otherwise every ~k/4 candidates (multiple of 32)
    for q, k, want in ((200, 1025, "cap"), (256, 129, "cap"), (257, 1025, 256), (600, 1025, 256), (200, 128, 32),
                       (600, 10, 32), (600, 2048, 512)):
        p = plan(50_037, 64, q, k)
        assert p["flush"] == (p["cap"] if want == "cap" else want), (q, k, p)
        assert p["cap"] == ((2 * k + p["bn"] + 31) // 32) * 32
    with pytest.raises(RuntimeError, match="k must be in"):
        plan(50_037, 64, 10, 2049)


@pytest.mark.parametrize("env,ld,q,want", [
    ({"B200REC_TOPK_V2": 0}, 64, 129, "nq2bn128"),
    ({"B200REC_TOPK_V2": 0}, 64, 600, "nq2bn128"),
    ({"B200REC_TOPK_V2": 0}, 256, 129, "nq2bn128"),
    ({"B200REC_TOPK_V2": 0}, 256, 600, "nq2bn128"),
    ({"B200REC_TOPK_V2": 0, "B200REC_TOPK_NQ": 1}, 64, 600, "bn256"),
    ({"B200REC_TOPK_V2": 1}, 128, 600, "pair1"),
    ({"B200REC_TOPK_V2": 2}, 128, 200, "pair2"),
    ({"B200REC_TOPK_V2": 2}, 64, 200, "pair2-ks1"),
])
def test_instantiation_knobs_force_what_they_name(env, ld, q, want):
    _need_148_sms()
    default = path_name(plan(50_037, ld, q, 10))
    assert default != want
    with topk_knobs(**env):
        assert path_name(plan(50_037, ld, q, 10)) == want
    assert path_name(plan(50_037, ld, q, 10)) == default


@pytest.mark.parametrize("N,Q,ld,k", [(300_000, 1500, 64, 20), (150_000, 4500, 64, 10)])
def test_schedule_knobs_on_the_work_split_shapes(N, Q, ld, k):
    """The shapes of test_flat_ip_topk_work_splits_bit_exact: by default the few leftover units idle."""
    _need_148_sms()
    assert decomposition(plan(N, ld, Q, k)) == "aligned-idle"
    for sched, want in (("0", "contiguous"), ("3", "aligned-working"), ("4", "aligned-idle")):
        with topk_knobs(B200REC_SCHED=sched):
            p = plan(N, ld, Q, k)
            assert decomposition(p) == want, (sched, p)
            if want == "contiguous":
                assert p["n_main"] == 0 and p["Tt"] == p["T"]
            if want == "aligned-working":
                assert p["Tmain"] + p["Tt"] == p["T"] and p["n_main"] == p["R"] * p["S"]
    assert decomposition(plan(N, ld, Q, k)) == "aligned-idle"


def test_sched_4_idles_leftover_units_on_a_long_scan():
    _need_148_sms()
    p = plan(20_000_000, 64, 1500, 20)
    assert p["W"] >= 6000 and decomposition(p) == "aligned-working"
    with topk_knobs(B200REC_SCHED=4):
        p4 = plan(20_000_000, 64, 1500, 20)
        assert p4["W"] == p["W"] and decomposition(p4) == "aligned-idle"
    assert decomposition(plan(20_000_000, 64, 1500, 20)) == "aligned-working"


def test_nosample_knob_and_reload_restore_the_sampling_pass():
    p = plan(50_037, 64, 300, 10)
    assert p["sample_m"] > 0
    with topk_knobs(B200REC_TOPK_NOSAMPLE=1):
        assert plan(50_037, 64, 300, 10)["sample_m"] == 0
    assert plan(50_037, 64, 300, 10) == p


def test_knobs_are_read_once_until_reloaded(monkeypatch):
    """A knob set without a reload does not change the plan of a shape already planned (or any other shape): the
    library reads the environment once; b200rec_debug_reload_env() is what makes a change take effect and, after the
    environment is restored, what brings the default plan back."""
    _need_148_sms()
    from topk_plan import reload
    base = plan(50_037, 128, 600, 10)
    assert path_name(base) == "pair2"
    monkeypatch.setenv("B200REC_TOPK_V2", "0")
    assert plan(50_037, 128, 600, 10) == base
    assert path_name(plan(50_037, 128, 601, 10)) == "pair2"
    reload()
    assert path_name(plan(50_037, 128, 600, 10)) == "nq2bn128"
    monkeypatch.delenv("B200REC_TOPK_V2")
    reload()
    assert plan(50_037, 128, 600, 10) == base


def test_topk_knobs_restores_on_failure():
    before = os.environ.get("B200REC_TOPK_V2")
    base = plan(50_037, 128, 600, 10)
    with pytest.raises(ZeroDivisionError):
        with topk_knobs(B200REC_TOPK_V2=0):
            assert path_name(plan(50_037, 128, 600, 10)) == "nq2bn128"
            1 / 0
    assert os.environ.get("B200REC_TOPK_V2") == before
    assert plan(50_037, 128, 600, 10) == base


def test_shards_argument_plans_the_pooled_sampling_density():
    """A row shard plans its sampling pass for the pooled catalogue of `shards` shards: a denser sample than alone."""
    p1, p2 = plan(300_000, 64, 300, 10), plan(300_000, 64, 300, 10, shards=2)
    assert p2["sample_m"] > p1["sample_m"] > 0
    assert path_name(p2) == path_name(p1)


def test_dimension_limit_is_reported_by_the_index_before_any_device_work():
    """fp32 storage keeps 3 bf16 pieces per value (ld = 3 * pad64(d)), so d > 192 has no plan; bf16 storage reaches
    d = 704.  The index and the engine refuse such a dimension when they are made, with the limit in the message."""
    from b200rec.retrieval import B200FlatIndex, FlatIPDeviceIndex, RetrievalEngine
    with pytest.raises(ValueError, match=r"192.*storage=.bf16.*704"):
        FlatIPDeviceIndex(256)
    with pytest.raises(ValueError, match=r"704"):
        FlatIPDeviceIndex(705, storage="bf16")
    with pytest.raises(ValueError, match=r"192"):
        B200FlatIndex({"dimension": 193})
    with pytest.raises(ValueError, match=r"192.*storage=.bf16"):
        RetrievalEngine({"index_type": "b200", "embedding_dim": 256})
    with pytest.raises(ValueError, match=r"704"):
        RetrievalEngine({"index_type": "b200", "embedding_dim": 768, "b200": {"storage": "bf16"}})
    assert RetrievalEngine({"index_type": "b200", "embedding_dim": 192}).index.dimension == 192
    assert RetrievalEngine({"index_type": "b200", "embedding_dim": 256, "b200": {"storage": "bf16"}}).index.dimension == 256
