"""Per-channel slider values (dspb_node_set_f32_channels) in planning mode (device -1, no GPU): argument checks, the plan
listing, the collapse of all-equal values to the shared case, and the scheduler's dataflow on random graphs with per-channel
fields.  The numeric side is tests/test_gpu_per_channel.py."""
import re

import numpy as np
import pytest

from dsp_stuff_b200 import GraphSpec
from dsp_stuff_b200 import signals as S
from dsp_stuff_b200.engine import Engine, EngineError
from tests.test_scheduler_fuzz import check_dataflow, parse_plan, plan_of

ERR_INVALID, ERR_UNKNOWN_NODE, ERR_UNKNOWN_PORT = -1, -2, -3

# every f32 field that may vary per channel (reverb.seconds may not)
FIELDS = {
    "gain": ["level"], "distort": ["level"], "overdrive": ["boost", "drive", "level"], "chebyshev": ["level_pos", "level_neg"],
    "biquad": ["a0", "a1", "a2", "b0", "b1", "b2"], "low_pass": ["ratio"], "high_pass": ["ratio"], "reverb": ["decay"],
    "mix": ["ratio"], "envelope": ["attack", "release"], "signal_gen": ["amplitude", "frequency"],
    "gate": ["threshold", "attack", "release"],
}


def planning_engine(g, channels, iir_mode=0):
    e = Engine(channels, block=128, max_samples=128 * 9, device=-1, iir_mode=iir_mode)
    g.apply(e)
    return e


def target(channels=8):
    return planning_engine(S.target_chain(64), channels)


def test_error_codes():
    C = 8
    e = target(C)
    v = np.linspace(0.5, 1.5, C, dtype=np.float32)
    with pytest.raises(EngineError) as ei:
        e.set_f32_channels(77, "level", v)
    assert ei.value.code == ERR_UNKNOWN_NODE
    with pytest.raises(EngineError) as ei:
        e.set_f32_channels(0, "no_such_field", v)
    assert ei.value.code == ERR_UNKNOWN_PORT
    with pytest.raises(EngineError) as ei:
        e.set_f32_channels(4, "taps", v)          # fir: no f32 fields at all
    assert ei.value.code == ERR_UNKNOWN_PORT
    with pytest.raises(EngineError) as ei:
        e.set_f32_channels(3, "seconds", v)       # ring length: one D per node
    assert ei.value.code == ERR_INVALID and "ring" in str(ei.value)
    for bad in (v[:-1], np.concatenate([v, v[:1]])):
        with pytest.raises(EngineError) as ei:
            e.set_f32_channels(0, "level", bad)
        assert ei.value.code == ERR_INVALID
    L = e._L
    assert L.dspb_node_set_f32_channels(e._h, 0, b"level", None, C) == ERR_INVALID
    assert L.dspb_node_set_f32_channels(e._h, 0, None, v.ctypes.data, C) == ERR_INVALID
    assert L.dspb_node_set_f32_channels(None, 0, b"level", v.ctypes.data, C) == ERR_INVALID


def test_every_supported_field_is_accepted():
    C = 4
    for t, fields in FIELDS.items():
        g = GraphSpec().node(0, t)
        e = planning_engine(g, C)
        for f in fields:
            e.set_f32_channels(0, f, np.arange(1, C + 1, dtype=np.float32))


def test_all_equal_values_are_the_shared_case_byte_for_byte():
    C = 16
    e = target(C)
    shared = e.describe_plan()
    for nid, field, val in [(0, "level", 2.0), (1, "level", 4.0), (3, "decay", 0.5)] + \
            [(2, k, v) for k, v in S.rbj_biquad("lp", 1000.0).items()]:
        e.set_f32_channels(nid, field, np.full(C, val, dtype=np.float32))
    e.compile()
    assert e.describe_plan() == shared
    # -0.0 and +0.0 differ in their bits: that is a per-channel field
    z = np.zeros(C, dtype=np.float32)
    z[3] = -0.0
    e.set_f32_channels(0, "level", z)
    e.compile()
    assert "per-channel[level]" in e.describe_plan()


def test_differing_values_are_marked_and_set_f32_restores_the_listing():
    C = 16
    e = target(C)
    shared = e.describe_plan()
    e.set_f32_channels(0, "level", np.linspace(0.5, 3.0, C))
    e.set_f32_channels(2, "b0", np.linspace(0.001, 0.01, C))
    e.set_f32_channels(3, "decay", np.linspace(0.1, 0.9, C))
    e.compile()
    plan = e.describe_plan()
    assert plan != shared
    assert "per-channel[level]" in plan and "per-channel[b0]" in plan and "per-channel[decay]" in plan
    assert "per-channel table 7 column(s)" in plan              # gain 1 + biquad 5 + comb 1
    ops = parse_plan(plan)[0][1]
    assert [o["code"] for o in ops] == [3, 13, 14, 20, 19, 11]
    assert ":c0" in plan and ":c1" in plan and ":c6" in plan
    # distort stays shared: its fast constant division is untouched
    assert "distort[SoftClip](acc, 4)  ;" in plan
    e.set_f32(0, "level", 2.0)
    e.set_f32(2, "b0", S.rbj_biquad("lp", 1000.0)["b0"])
    e.compile()
    assert "per-channel[decay]" in e.describe_plan() and "per-channel[level]" not in e.describe_plan()
    e.set_f32(3, "decay", 0.5)
    e.compile()
    assert e.describe_plan() == shared


def test_linked_control_port_overrides_per_channel_values():
    C = 4
    g = (GraphSpec().node(10, "input").node(11, "input").node(12, "output").node(0, "gain")
         .link(10, "out", 0, "in").link(11, "out", 0, "level").link(0, "out", 12, "in"))
    e = planning_engine(g, C)
    shared = e.describe_plan()
    e.set_f32_channels(0, "level", np.arange(1, C + 1, dtype=np.float32))   # channel 0 keeps the default 1.0
    e.compile()
    assert e.describe_plan() == shared


def test_scan_mode_keeps_a_per_channel_biquad_exact():
    C = 256
    g = S.config2()
    e = planning_engine(g, C, iir_mode=1)
    assert e.describe_plan().count("time-parallel scan") == 2
    e.set_f32_channels(0, "b0", np.linspace(0.001, 0.002, C))
    e.compile()
    plan = e.describe_plan()
    assert "exact (per-channel coefficients) per-channel[b0]" in plan
    # all or nothing per segment: the other biquad of the segment is exact as well
    assert plan.count("[exact after all: another recurrence of this segment stays sequential]") == 1


def test_per_channel_filter_does_not_count_toward_the_scan_table_limit():
    """Ten low-pass filters, iir_mode = 1: four scan tables per Program cut the chain into three segments.  With one of the
    ten per-channel, nine qualify and the per-channel one never occupies a table."""
    C = 256
    g = GraphSpec().node(100, "input").node(101, "output")
    prev = 100
    for i in range(10):
        g.node(i, "low_pass", ratio=0.5 + 0.04 * i)
        g.link(prev, "out", i, "in")
        prev = i
    g.link(prev, "out", 101, "in")
    e = planning_engine(g, C, iir_mode=1)
    assert e.describe_plan().count("fused segment:") == 3
    e.set_f32_channels(4, "ratio", np.linspace(0.3, 0.6, C))
    e.compile()
    plan = e.describe_plan()
    check_dataflow(plan, 1)
    assert plan.count("exact (per-channel coefficients)") == 1


def test_table_overflow_cuts_the_segment():
    """33 gains with per-channel levels: one table holds 32 columns, so the chain is cut, not refused."""
    C = 64
    g = GraphSpec().node(100, "input").node(101, "output")
    prev = 100
    for i in range(33):
        g.node(i, "gain", level=1.0 + i / 64)
        g.link(prev, "out", i, "in")
        prev = i
    g.link(prev, "out", 101, "in")
    e = planning_engine(g, C)
    assert e.describe_plan().count("fused segment:") == 1
    for i in range(33):
        e.set_f32_channels(i, "level", np.linspace(0.5, 1.5, C) + i)
    e.compile()
    plan = e.describe_plan()
    check_dataflow(plan, 1)
    assert plan.count("fused segment:") == 2
    assert plan.count("per-channel[level]") == 33
    for k in map(int, re.findall(r"per-channel table (\d+) column", plan)):
        assert k <= 32


@pytest.mark.parametrize("seed", range(30))
def test_random_graphs_with_per_channel_fields_lower_with_sound_dataflow(seed):
    rng = np.random.default_rng(5000 + seed)
    g = S.random_graph(seed, None if seed < 15 else 10 + seed)
    C = 64 if seed % 2 else 4096
    shared = plan_of(g, C)
    e = planning_engine(g, C, iir_mode=seed % 3 == 0)
    n_pc = 0
    for nd in g.nodes:
        for f in FIELDS.get(nd.typename, []):
            if rng.uniform() < 0.5:
                e.set_f32_channels(nd.id, f, rng.uniform(0.0, 1.0, C).astype(np.float32))
                n_pc += 1
    e.compile()
    plan = e.describe_plan()
    check_dataflow(plan, 2)
    if n_pc == 0:
        assert plan == shared or seed % 3 == 0
