"""The two-instruction constant division (exact_math.cuh div_const2: q = fma(a, zh, a*zl)) on the device: proof by
enumeration of all 2^32 dividends per divisor, the engine's tier choice, and chunks that must take the IEEE fallback
(zeros of either sign, subnormals, +-2^90, infinities, NaN) through the compiled target chain and the interpreter."""
import os
import subprocess

import numpy as np
import pytest

from dsp_stuff_b200 import GraphSpec
from dsp_stuff_b200 import signals as S
from tests.test_const_div2_planning import lowered_tiers
from tests.test_gpu_parity import run_both
from tests.util import assert_bit_exact

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def fan_in_divisors(links=8):
    nf, out = np.float32(0.0001), []
    for _ in range(links):
        nf = np.float32(nf + np.float32(1.0))
        out.append(float(nf))
    return out


def test_div_const2_matches_ieee_for_every_f32_dividend(tmp_path):
    exe = str(tmp_path / "div2_exhaustive")
    from dsp_stuff_b200.build import _nvcc

    subprocess.check_call([_nvcc(), "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-o", exe,
                           os.path.join(ROOT, "tests", "cuda", "div2_exhaustive.cu")])
    # the fan-in averages of 1..8 links, SoftClip's /3 (compiled in as a constant), Distort levels, and three divisors
    # far from 1 (0.3 fails Markstein's form)
    divisors = fan_in_divisors() + [3.0, 4.0, 0.5, 16.0, 29.99, 7.0, 1.5, 1e-3, 0.3, 1e3]
    out = subprocess.run([exe] + [repr(d) for d in divisors], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stdout + out.stderr
    lines = [l.split() for l in out.stdout.strip().splitlines()]
    assert len(lines) == len(divisors)
    for b, mism, flagged in lines:
        assert int(mism) == 0, f"divisor {b}: {mism} mismatching dividends"
        # the window 2^-96 <= |a| <= 2^96 leaves 64 of 256 binades, zeros, infinities and NaNs to the fallback
        assert int(flagged) < 0.30 * 2 ** 32, (b, flagged)


def test_engine_verifies_and_lists_the_two_instruction_tier():
    from dsp_stuff_b200.engine import Engine

    e = Engine(64, block=128, max_samples=1024)
    S.target_chain(64).apply(e)
    e.process(S.noise(64, 1024))
    ops = lowered_tiers(e.describe_plan())[0]
    assert [o[1] for o in ops] == [None] + ["mul-fma"] * 5
    assert [o[2] for o in ops] == [None, None, "mul-fma", None, None, None]


SPECIALS = np.array([0.0, -0.0, 1e-40, -1e-42, 2.0 ** -126, 2.0 ** 90, -2.0 ** 90, np.inf, -np.inf, np.nan, 2.0 ** 127],
                    dtype=np.float32)


def with_specials(C, n, seed):
    """noise with, per channel, a few 8-sample chunks that each hold one special value (channel c gets special c % k, so
    one NaN or infinity poisons only its own channel's recurrences)"""
    x = S.noise(C, n, seed=seed)
    rng = np.random.default_rng(seed)
    for c in range(C):
        for chunk in rng.choice(n // 8, size=4, replace=False):
            x[c, chunk * 8 + int(rng.integers(8))] = SPECIALS[c % len(SPECIALS)]
    x[:, 1024:1032] = 0.0                  # one whole chunk of zeros in every channel
    return x


def assert_bits(got, ref, what):
    got = np.asarray(got, np.float32)
    ref = np.asarray(ref, np.float32)
    same = (got.view(np.uint32) == ref.view(np.uint32)) | (np.isnan(got) & np.isnan(ref))   # zero signs included
    assert same.all(), f"{what}: {np.count_nonzero(~same)} samples differ, first at {tuple(np.argwhere(~same)[0])}"


@pytest.mark.parametrize("name, spec", [
    ("target", S.target_chain(64)),    # compiled chain in the warp-specialised kernel (direct FIR: bit-exact)
    ("hardclip_29.99", GraphSpec().node(10, "input").node(11, "output").node(0, "gain", level=3.0)
     .node(1, "distort", mode="HardClip", level=29.99).link(10, "out", 0, "in").link(0, "out", 1, "in")
     .link(1, "out", 11, "in")),      # interpreter
])
def test_fallback_chunks_match_the_oracle_bit_for_bit(oracle_mod, name, spec):
    C, n = 64, 4096
    x = with_specials(C, n, seed=11)
    got, ref, _ = run_both(oracle_mod, spec, x, chunks=[2048, 2048])
    if name == "target":
        assert_bit_exact(got[0], ref[0], name)    # the direct FIR's f64 sums: the suite's bit-exact (-0.0 == +0.0)
    else:
        assert_bits(got[0], ref[0], name)
