"""Exhaustive proof-by-enumeration that the 3-instruction constant division used for the fan-in average
(node.rs:189-191) and the clip shapers is bit-identical to IEEE division: all 2^32 dividends per divisor."""
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_div_const_matches_ieee_for_every_f32_dividend(tmp_path):
    exe = str(tmp_path / "div_exhaustive")
    from dsp_stuff_b200.build import _nvcc   # the compiler the library is built with, also when nvcc is not on PATH

    subprocess.check_call([_nvcc(), "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-o", exe,
                           os.path.join(ROOT, "tests", "cuda", "div_exhaustive.cu")])
    nf = np.float32(0.0001)
    divisors = []
    for _ in range(8):                      # 1..8 links into one port
        nf = np.float32(nf + np.float32(1.0))
        divisors.append(float(nf))
    divisors += [3.0, 4.0, 0.5, 16.0, 29.99, 7.0, 1.5]   # SoftClip's /3 and some Distort levels
    # (the engine re-runs this very enumeration on the device for every divisor it meets and uses
    #  IEEE division if it finds a single mismatch: engine.cpp div_const_ok / verify_const_div)
    out = subprocess.run([exe] + [repr(d) for d in divisors], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr
    lines = [l.split() for l in out.stdout.strip().splitlines()]
    assert len(lines) == len(divisors)
    for b, mism, flagged in lines:
        assert int(mism) == 0, f"divisor {b}: {mism} mismatching dividends"
        # only tiny / huge / non-finite quotients may take the slow path (< 30 % of all bit patterns)
        assert int(flagged) < 0.35 * 2 ** 32, (b, flagged)
