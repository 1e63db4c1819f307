"""Per-channel slider values (dspb_node_set_f32_channels) on the GPU against the CPU oracle.

Reference: the channels are grouped by their parameter set and one Oracle per group runs exactly the channels that hold it,
with plain set_f32.  FMA-free nodes compare bit for bit, the libm ones (Tanh, Sin, Atan, Fuzz, overdrive, chebyshev, Sine)
and the FFT FIR within the parity tolerance.
"""
import re

import numpy as np
import pytest

from dsp_stuff_b200 import GraphSpec
from dsp_stuff_b200 import signals as S
from tests.util import assert_audio_close, assert_bit_exact, make_oracle

pytestmark = pytest.mark.gpu
FIR_FFT, FIR_DIRECT = 0, 1


def f32(v):
    return np.asarray(v, dtype=np.float32)


class Grouped:
    """One Oracle per distinct parameter set.  values: {(node, field): [C] array}.  set() applies a later setter to both."""

    def __init__(self, oracle_mod, spec, values, C):
        keys = sorted(values)
        rows = np.stack([f32(values[k]).view(np.uint32) for k in keys], axis=1) if keys else np.zeros((C, 0), np.uint32)
        self.groups = {}
        for c in range(C):
            self.groups.setdefault(rows[c].tobytes(), []).append(c)
        self.C = C
        self.parts = []
        for idx in self.groups.values():
            idx = np.array(idx)
            o = make_oracle(oracle_mod, spec, len(idx))
            for k in keys:
                o.set_f32(k[0], k[1], float(f32(values[k])[idx[0]]))
            self.parts.append((idx, o))

    def set(self, node, field, values):
        """values: [C], constant on every group (else the grouping would have to change)."""
        v = f32(values)
        for idx, o in self.parts:
            assert np.all(v[idx].view(np.uint32) == v[idx[0]].view(np.uint32))
            o.set_f32(node, field, float(v[idx[0]]))

    def process(self, xs, n=None):
        outs = None
        for idx, o in self.parts:
            r = o.process([x[idx] for x in xs]) if xs else o.process_n(n)
            if outs is None:
                outs = [np.zeros((self.C, r[0].shape[1]), np.float32) for _ in r]
            for a, b in zip(outs, r):
                a[idx] = b
        return outs


def engine(spec, C, n, fir_mode=FIR_DIRECT, **kw):
    from dsp_stuff_b200.engine import Engine

    e = Engine(C, block=128, max_samples=n, fir_mode=fir_mode, **kw)
    spec.apply(e)
    return e


def apply_pc(e, values):
    for (node, field), v in values.items():
        e.set_f32_channels(node, field, v)


def spread(vals, C, k=0):
    """Channel c gets vals[(c * (2k + 1) + k) % len(vals)]: groups interleave across channels and across fields."""
    vals = f32(vals)
    c = np.arange(C)
    return vals[(c * (2 * k + 1) + k) % len(vals)]


def compare(got, ref, exact, what):
    for i, (g, r) in enumerate(zip(got, ref)):
        if exact:
            assert_bit_exact(g, r, f"{what} out{i}")
        else:
            assert_audio_close(g, r, what=f"{what} out{i}")


# ---- every supported field: C = 64, 8 distinct values per field, two calls with state carried ------------------------
RBJ = [S.rbj_biquad("lp", f) for f in (300.0, 500.0, 800.0, 1200.0, 2000.0, 3000.0, 5000.0, 9000.0)]
A0 = [1.0, 2.0, 0.5, 1.5, 1.0, 3.0, 0.8, 1.25]
FIELD_VALUES = {
    "gain": {"level": [0.0, 0.5, 1.0, 2.5, -1.0, 12.0, 0.001, 3.0]},
    "distort": {"level": [0.0, 0.0005, 0.001, 1.0, 4.0, 7.3, 35.0, -2.0]},     # 0 and < 0.001: the early-out; 35: out of range
    "overdrive": {"boost": [0.0, 1.0, 5.0, 30.0, 40.0, 2.0, 3.0, 10.0], "drive": [0.0, 0.25, 0.5, 1.0, 1.5, 0.1, 0.9, 0.7],
                  "level": [0.0, 0.0005, 0.5, 1.0, 2.0, 0.3, 0.8, 0.1]},
    "chebyshev": {"level_pos": [0.0, 0.0005, 1.0, 5.0, 50.0, 60.0, 2.0, 0.3], "level_neg": [0.3, 2.0, 0.0, 60.0, 1.0, 0.0005, 5.0, 50.0]},
    "biquad": {k: [r[k] * a for r, a in zip(RBJ, A0)] for k in ("a0", "a1", "a2", "b0", "b1", "b2")},   # a0 != 1
    "low_pass": {"ratio": [0.0, 0.1, 0.5, 0.9, 0.99, 0.999, 0.3, -0.2]},
    "high_pass": {"ratio": [0.0, 0.1, 0.5, 0.9, 0.99, 0.999, 0.3, -0.2]},
    "reverb": {"decay": [0.0, 0.1, 0.5, 0.9, 1.0, 1.1, -0.5, 0.25]},
    "mix": {"ratio": [0.0, 0.25, 0.5, 1.0, -0.5, 1.5, 0.75, 0.1]},
    "envelope": {"attack": [0.0, 1.0, 5.0, 50.0, 400.0, 1000.0, 2000.0, 0.5], "release": [0.0, 3.0, 10.0, 100.0, 400.0, 1000.0, 0.5, 2.0]},
    "gate": {"threshold": [0.0, 0.05, 0.1, 0.2, 0.3, 0.5, 1.0, -1.0], "attack": [0.0, 1.0, 5.0, 50.0, 3.0, 10.0, 2.0, 0.5],
             "release": [0.0, 3.0, 10.0, 100.0, 400.0, 150.0, 0.5, 2.0]},
    "signal_gen": {"amplitude": [-1.0, -0.5, 0.0, 0.25, 0.5, 1.0, 2.0, 0.75],
                   "frequency": [0.1, 50.0, 100.0, 441.0, 1000.0, 5000.0, 20000.0, 30000.0]},
}
CASES = [("gain", {}, True), ("distort", dict(mode="HardClip"), True), ("distort", dict(mode="SoftClip"), True),
         ("distort", dict(mode="RecipSoftClip"), True), ("distort", dict(mode="Square"), True),
         ("distort", dict(mode="Chebyshev4"), True), ("distort", dict(mode="Tanh"), False), ("distort", dict(mode="Sin"), False),
         ("distort", dict(mode="Atan"), False), ("distort", dict(mode="Fuzz"), False), ("overdrive", {}, False),
         ("chebyshev", {}, False), ("biquad", {}, True), ("low_pass", {}, True), ("high_pass", {}, True),
         ("reverb", dict(seconds=0.01), True), ("mix", {}, True), ("envelope", {}, True), ("gate", {}, True),
         ("signal_gen", dict(mode="Triangle"), True), ("signal_gen", dict(mode="Square"), True),
         ("signal_gen", dict(mode="Sine"), False)]


def single_node_graph(t, params):
    g = GraphSpec().node(0, t, **params).node(11, "output")
    if t == "signal_gen":
        return g.link(0, "out", 11, "in")
    g.node(10, "input")
    if t == "mix":
        g.node(1, "gain", level=-0.7).link(10, "out", 1, "in").link(10, "out", 0, "a").link(1, "out", 0, "b")
    else:
        g.link(10, "out", 0, "in")
    return g.link(0, "out", 11, "in")


@pytest.mark.parametrize("t,params,exact", CASES, ids=[f"{t}-{p.get('mode', '')}" for t, p, _ in CASES])
def test_every_field_against_grouped_oracle(oracle_mod, t, params, exact):
    C, n = 64, 128 * 24
    g = single_node_graph(t, params)
    fv = FIELD_VALUES[t]
    if params.get("mode") == "Fuzz":
        # Fuzz has no early-out, and at tiny levels 1 - exp(-q) cancels: the 1-2 ulp libm difference grows past the bar
        fv = {"level": [0.0, 0.1, 0.5, 1.0, 4.0, 7.3, 35.0, -2.0]}
    values = {(0, f): spread(v, C, k) for k, (f, v) in enumerate(fv.items())}
    if t == "biquad":   # the six coefficients of one filter belong together
        values = {(0, f): spread(v, C) for f, v in FIELD_VALUES[t].items()}
    ref_eng = Grouped(oracle_mod, g, values, C)
    e = engine(g, C, n // 2)
    apply_pc(e, values)
    x = S.noise(C, n)
    for call in range(2):
        part = slice(call * n // 2, (call + 1) * n // 2)
        if t == "signal_gen":
            got, ref = e.process([], n // 2), ref_eng.process([], n // 2)
        else:
            got, ref = e.process([x[:, part]]), ref_eng.process([x[:, part]])
        if exact:
            compare(got, ref, True, f"{t} call {call}")
        else:  # per group: some groups are all zero (amplitude 0) or non-finite (Fuzz at level 0: 0 / 0), like the reference
            for idx, _ in ref_eng.parts:
                close_group(got[0][idx], ref[0][idx], f"{t} call {call} group {idx[0]}")


def close_group(g, r, what):
    fin = np.isfinite(r)
    assert np.array_equal(fin, np.isfinite(g)), f"{what}: non-finite samples differ"
    if np.max(np.abs(r[fin]), initial=0.0) == 0.0:
        assert_bit_exact(g[fin], r[fin], what)
    else:
        assert_audio_close(g[fin], r[fin], what=what)


# ---- launch shapes -------------------------------------------------------------------------------------------------
def target_values(C):
    lp = [S.rbj_biquad("lp", f) for f in np.linspace(500.0, 4000.0, 8)]
    v = {(0, "level"): spread([0.5, 1.0, 1.5, 2.0, 2.5, 3.0, 0.25, 4.0], C, 1),
         (1, "level"): spread([0.0, 0.5, 1.0, 2.0, 4.0, 6.0, 8.0, 3.3], C, 2),
         (3, "decay"): spread([0.1, 0.2, 0.3, 0.4, 0.5, 0.6, 0.7, 0.8], C, 3)}
    for k in ("a1", "a2", "b0", "b1", "b2"):
        v[(2, k)] = spread([r[k] for r in lp], C)
    return v


@pytest.mark.parametrize("C,fir_mode,n_taps,n", [(64, FIR_DIRECT, 256, 128 * 160), (4096, FIR_FFT, 64, 2048)])
def test_target_chain(oracle_mod, C, fir_mode, n_taps, n):
    g = S.target_chain(n_taps)
    values = target_values(C)
    ref_eng = Grouped(oracle_mod, g, values, C)
    e = engine(g, C, n // 2, fir_mode=fir_mode)
    apply_pc(e, values)
    x = S.noise(C, n)
    for call in range(2):
        part = slice(call * n // 2, (call + 1) * n // 2)
        compare(e.process([x[:, part]]), ref_eng.process([x[:, part]]), fir_mode == FIR_DIRECT, f"target C={C} call {call}")


@pytest.mark.parametrize("one_pole", [False, True])
def test_config2_two_recurrence_kernel(oracle_mod, one_pole):
    C, n = 256, 128 * 64
    g = S.config2(one_pole=one_pole)
    if one_pole:
        values = {(0, "ratio"): spread([0.5, 0.8, 0.9, 0.95, 0.99, 0.7, 0.6, 0.85], C, 1),
                  (1, "ratio"): spread([0.9, 0.95, 0.99, 0.999, 0.5, 0.8, 0.97, 0.93], C, 2)}
    else:
        lp = [S.rbj_biquad("lp", f) for f in np.linspace(500.0, 4000.0, 8)]
        hp = [S.rbj_biquad("hp", f) for f in np.linspace(100.0, 800.0, 8)]
        values = {}
        for k in ("a1", "a2", "b0", "b1", "b2"):
            values[(0, k)] = spread([r[k] for r in lp], C, 0)
            values[(1, k)] = spread([r[k] for r in hp], C, 1)
    ref_eng = Grouped(oracle_mod, g, values, C)
    e = engine(g, C, n // 2)
    apply_pc(e, values)
    x = S.noise(C, n)
    for call in range(2):
        part = slice(call * n // 2, (call + 1) * n // 2)
        compare(e.process([x[:, part]]), ref_eng.process([x[:, part]]), True, f"config2 one_pole={one_pole} call {call}")


def test_config5_interpreter_with_vregs(oracle_mod):
    C, n = 64, 128 * 120
    g = S.config5(64)
    lp = [S.rbj_biquad("lp", f) for f in np.linspace(500.0, 4000.0, 8)]
    values = {(0, "level"): spread([0.5, 1.0, 1.5, 2.0, 2.5, 3.0, 0.25, 4.0], C, 1),
              (1, "level"): spread([0.0, 0.5, 1.0, 2.0, 4.0, 6.0, 8.0, 3.3], C, 2),
              (6, "decay"): spread([0.1, 0.2, 0.3, 0.4, 0.5, 0.6, 0.7, 0.8], C, 3),
              (8, "ratio"): spread([0.0, 0.2, 0.4, 0.5, 0.6, 0.8, 1.0, 0.3], C, 4)}
    for k in ("a1", "a2", "b0", "b1", "b2"):
        values[(3, k)] = spread([r[k] for r in lp], C)
    ref_eng = Grouped(oracle_mod, g, values, C)
    e = engine(g, C, n // 2)
    apply_pc(e, values)
    x = S.noise(C, n)
    for call in range(2):
        part = slice(call * n // 2, (call + 1) * n // 2)
        compare(e.process([x[:, part]]), ref_eng.process([x[:, part]]), False, f"config5 call {call}")
    plan = e.describe_plan()      # lowered at the first call
    assert re.search(r"[1-9]\d* smem vregs.*per-channel table", plan), plan


def _device_process(e, xs, C, n):
    import torch

    ins = [torch.from_numpy(x).cuda() for x in xs]
    outs = [torch.empty((C, n), dtype=torch.float32, device="cuda") for _ in range(e._n_out)]
    e.process_device(ins, outs, n)
    torch.cuda.synchronize()
    return [o.cpu().numpy() for o in outs]


@pytest.mark.parametrize("env", [("DSPB_FORCE_G", "1"), ("DSPB_FORCE_G", "4"), ("DSPB_FORCE_G", "16"),
                                 ("DSPB_FORCE_G", "32"), ("DSPB_CHUNKS", "4")])
@pytest.mark.parametrize("path", ["host", "device"])
def test_launch_variants(oracle_mod, monkeypatch, env, path):
    monkeypatch.setenv(*env)
    C, n = 256, 128 * 32
    g = S.target_chain(64)
    values = target_values(C)
    ref_eng = Grouped(oracle_mod, g, values, C)
    e = engine(g, C, n // 2)
    apply_pc(e, values)
    x = S.noise(C, n)
    for call in range(2):
        part = np.ascontiguousarray(x[:, call * n // 2:(call + 1) * n // 2])
        got = e.process([part]) if path == "host" else _device_process(e, [part], C, n // 2)
        compare(got, ref_eng.process([part]), True, f"{env} {path} call {call}")


# ---- equivalences --------------------------------------------------------------------------------------------------
def test_row_equals_an_engine_with_that_rows_values():
    C, n = 64, 128 * 40
    g = S.target_chain(64)
    values = target_values(C)
    e = engine(g, C, n)
    apply_pc(e, values)
    x = S.noise(C, n)
    got = e.process([x])[0]
    for c in (0, 13, 63):
        s = engine(g, C, n)
        for (node, field), v in values.items():
            s.set_f32(node, field, float(v[c]))
        assert_bit_exact(got[c], s.process([x])[0][c], f"row {c}")


@pytest.mark.parametrize("fir_mode", [FIR_DIRECT, FIR_FFT])
def test_all_equal_values_collapse_to_the_shared_case(fir_mode):
    C, n = 4096, 2048
    g = S.target_chain(256)
    shared = engine(g, C, n, fir_mode=fir_mode)
    pc = engine(g, C, n, fir_mode=fir_mode)
    for nid, field, val in [(0, "level", 2.0), (1, "level", 4.0), (3, "decay", 0.5)] + \
            [(2, k, v) for k, v in S.rbj_biquad("lp", 1000.0).items()]:
        pc.set_f32_channels(nid, field, np.full(C, val, dtype=np.float32))
    x = S.noise(C, n)
    a, b = shared.process([x])[0], pc.process([x])[0]
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    assert shared.kernel_launches == pc.kernel_launches
    assert shared.describe_plan() == pc.describe_plan()


def test_setter_semantics(oracle_mod):
    """A per-channel biquad change resets the filter state, a per-channel decay change resets the ring, set_f32 returns a
    field to shared; the oracle groups get set_f32 at the same points."""
    C, n = 64, 128 * 100
    g = S.config3()
    lp = [S.rbj_biquad("lp", f) for f in np.linspace(500.0, 4000.0, 8)]
    values = {(3, "decay"): spread([0.1, 0.2, 0.3, 0.4, 0.5, 0.6, 0.7, 0.8], C)}
    for k in ("a1", "a2", "b0", "b1", "b2"):
        values[(2, k)] = spread([r[k] for r in lp], C)
    ref_eng = Grouped(oracle_mod, g, values, C)
    e = engine(g, C, n)
    apply_pc(e, values)
    x = S.noise(C, 3 * n)

    def set_both(node, field, v):
        e.set_f32_channels(node, field, v)
        ref_eng.set(node, field, v)

    for call in range(3):
        if call == 1:   # new per-channel coefficients: every channel's filter state starts from zero
            set_both(2, "b0", spread([r["b0"] * 0.5 for r in lp], C))
        if call == 2:   # new per-channel decay: the ring is refreshed (zero-filled)
            set_both(3, "decay", spread([0.9, 0.8, 0.7, 0.6, 0.5, 0.4, 0.3, 0.2], C))
        part = x[:, call * n:(call + 1) * n]
        compare(e.process([part]), ref_eng.process([part]), True, f"setter call {call}")
    e.set_f32(3, "decay", 0.45)     # shared again
    ref_eng.set(3, "decay", np.full(C, 0.45, np.float32))
    compare(e.process([x[:, :n]]), ref_eng.process([x[:, :n]]), True, "after set_f32")
    plan = e.describe_plan()
    assert "per-channel[decay]" not in plan and "per-channel[a1,a2,b0,b1,b2]" in plan


def test_scan_mode_per_channel_biquad_exact_shared_one_scans(oracle_mod):
    C, n = 256, 128 * 64
    g = (GraphSpec().node(10, "input").node(11, "output").node(12, "output")
         .node(0, "biquad", **S.rbj_biquad("lp", 1000.0)).node(1, "fir", mode="Balanced", taps=[1.0])
         .node(2, "biquad", **S.rbj_biquad("lp", 1000.0))
         .link(10, "out", 0, "in").link(0, "out", 11, "in").link(0, "out", 1, "in").link(1, "out", 2, "in").link(2, "out", 12, "in"))
    lp = [S.rbj_biquad("lp", f) for f in np.linspace(500.0, 4000.0, 8)]
    values = {(0, k): spread([r[k] for r in lp], C) for k in ("a1", "a2", "b0", "b1", "b2")}
    ref_eng = Grouped(oracle_mod, g, values, C)
    e = engine(g, C, n, iir_mode=1)
    apply_pc(e, values)
    x = S.noise(C, n)
    got, ref = e.process([x]), ref_eng.process([x])
    plan = e.describe_plan()
    assert "exact (per-channel coefficients)" in plan and plan.count("time-parallel scan") == 1, plan
    assert_bit_exact(got[0], ref[0], "per-channel biquad (exact)")
    assert_audio_close(got[1], ref[1], what="shared biquad (scan)")


def test_shards_equal_the_whole_run():
    from dsp_stuff_b200.shard import channel_range

    C, n = 256, 128 * 40
    g = S.target_chain(64)
    values = target_values(C)
    x = S.noise(C, n)
    whole = engine(g, C, n)
    apply_pc(whole, values)
    ref = whole.process([x])[0]
    for r in range(2):
        lo, hi = channel_range(r, 2, C)
        s = engine(g, hi - lo, n)
        apply_pc(s, {k: v[lo:hi] for k, v in values.items()})
        assert_bit_exact(s.process([np.ascontiguousarray(x[lo:hi])])[0], ref[lo:hi], f"shard {r}")


def test_node_process(oracle_mod):
    C, n = 64, 128 * 16
    g = GraphSpec().node(0, "biquad")
    lp = [S.rbj_biquad("lp", f) for f in np.linspace(500.0, 4000.0, 8)]
    values = {(0, k): spread([r[k] for r in lp], C) for k in ("a1", "a2", "b0", "b1", "b2")}
    ref_eng = Grouped(oracle_mod, g, values, C)
    e = engine(g, C, n)
    apply_pc(e, values)
    x = S.noise(C, 2 * n)
    for call in range(2):
        part = x[:, call * n:(call + 1) * n]
        got = e.node_process(0, [part])[0]
        ref = np.zeros_like(got)
        for idx, o in ref_eng.parts:
            ref[idx] = o.node_process(0, [part[idx]])[0]
        assert_bit_exact(got, ref, f"node_process call {call}")


def test_async_host_path_matches_blocking():
    C, n = 256, 128 * 16
    g = S.config3()
    x = [S.noise(C, n, seed=s) for s in range(3)]
    levels = [spread([0.5, 1.0, 2.0, 3.0], C, k) for k in range(3)]

    def run(wait):
        import torch

        e = engine(g, C, n)
        outs = []
        for k in range(3):
            e.set_f32_channels(0, "level", levels[k])
            xi = torch.from_numpy(x[k]).pin_memory()
            yo = torch.empty((C, n), dtype=torch.float32).pin_memory()
            e.process_host([xi], [yo], n, wait=wait)
            outs.append((xi, yo))
        e.sync()
        return [yo.numpy().copy() for _, yo in outs]

    for a, b in zip(run(True), run(False)):
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
