"""The plan listing names how every constant division runs (csrc/engine.cpp div_tier): the fan-in divisor (`:nf=`) and a
Distort's scalar level (`:div=`) on the `lowered:` line.  Planning mode (device -1, no GPU) verifies nothing, so a fast tier
is marked `?`; the device side is tests/test_gpu_const_div2.py."""
import re

import numpy as np

from dsp_stuff_b200 import signals as S
from dsp_stuff_b200.engine import Engine
from tests.test_oracle_kat import single


def lowered_tiers(plan):
    """-> per fused step, per op: (code, nf tier or None, div tier or None)"""
    out = []
    for line in plan.splitlines():
        if line.startswith("    lowered:"):
            ops = []
            for tok in line.split()[1:]:
                parts = tok.split(":")
                nf = next((p[3:] for p in parts if p.startswith("nf=")), None)
                dv = next((p[4:] for p in parts if p.startswith("div=")), None)
                ops.append((int(parts[0]), nf, dv))
            out.append(ops)
    return out


def plan(g, channels=8):
    e = Engine(channels, block=128, max_samples=128 * 9, device=-1)
    g.apply(e)
    return e, e.describe_plan()


def test_target_chain_lists_every_division_with_its_tier():
    _, p = plan(S.target_chain(64))
    ops = lowered_tiers(p)[0]
    # LOADG, GAIN, DISTORT(SoftClip), BIQUAD, COMB, STOREG: five fan-in divisions by 1.0001 and the level 4
    assert [o[1] for o in ops] == [None] + ["mul-fma?"] * 5, p
    assert [o[2] for o in ops] == [None, None, "mul-fma?", None, None, None], p


def test_divisor_outside_the_two_instruction_range_is_listed_as_markstein():
    for level, tier in [(2.0 ** 20, "mul-fma?"), (2.0 ** 21, "markstein?"), (2.0 ** -21, "markstein?"), (1e-31, "ieee")]:
        _, p = plan(single("distort", mode="HardClip", level=level))
        dist = [o for o in lowered_tiers(p)[0] if o[2] is not None]
        assert len(dist) == 1 and dist[0][2] == tier, (level, p)


def test_per_channel_level_divides_with_ieee_division():
    C = 8
    e, _ = plan(S.target_chain(64), C)
    e.set_f32_channels(1, "level", np.linspace(1.0, 4.0, C, dtype=np.float32))
    e.compile()
    p = e.describe_plan()
    dist = [o for o in lowered_tiers(p)[0] if o[2] is not None]
    assert len(dist) == 1 and dist[0][2] == "ieee", p
    assert "per-channel[level]" in p


def test_fan_in_of_several_links_lists_its_divisor_tier():
    _, p = plan(S.config5(64))
    tiers = {t for step in lowered_tiers(p) for _, t, _ in step if t is not None}
    assert tiers == {"mul-fma?"}, p
    assert re.search(r"acc /= 2\.00010014", p)
