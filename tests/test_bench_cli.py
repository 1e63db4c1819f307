"""bench.py contract checks: the reference arm (the oracle port on the host cores) needs no GPU; --dump-outputs does."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from dsp_stuff_b200 import signals as S
from tests.util import assert_bit_exact

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=600, env=e)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout   # ONE JSON line on stdout, nothing else
    return json.loads(lines[0])


def test_reference_arm_prints_the_contract_line():
    d = run_bench("--impl", "reference", "--steps", "2", "--warmup", "1", "--workload", "config3")
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "channel_samples_per_sec" and d["higher_is_better"] is True
    assert d["vs_baseline"] is None and d["dtype"] == "f32" and d["data"] == "synthetic"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"] == "config3" and d["config"]["scaling"] == "strong" and d["config"]["channels"] == 1024
    assert d["value"] > 0


def test_reference_arm_other_ranks_exit_quietly():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=300, env=dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1"))
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_strong_scaling_shards_are_what_both_arms_report():
    d = run_bench("--impl", "reference", "--gpus", "8", "--steps", "1", "--warmup", "0", env={"RANK": "0", "WORLD_SIZE": "8"})
    assert d["config"]["channels"] == 4096 and d["config"]["channels_per_gpu"] == 512 and d["scaling"] == "strong"
    d = run_bench("--impl", "reference", "--gpus", "8", "--steps", "1", "--warmup", "0", "--scaling", "weak", env={"RANK": "0", "WORLD_SIZE": "8"})
    assert d["config"]["channels"] == 8 * 4096 and d["config"]["channels_per_gpu"] == 4096 and d["scaling"] == "weak"


@pytest.mark.gpu
def test_dump_outputs_is_the_last_timed_step(tmp_path):
    """--steps K --warmup 3: the dumped array is the engine's output of its 3 + K-th call on the seeded bench input."""
    from dsp_stuff_b200.engine import Engine

    C, n, steps = 8, 2048, 4
    d = run_bench("--workload", "config3", "--channels", str(C), "--blocks-per-step", "2", "--steps", str(steps), "--warmup", "3",
                  "--no-cpu-baseline", "--no-e2e", "--no-parity", "--no-block-calls", "--no-scan-side", "--sustain-seconds", "0",
                  "--dump-outputs", str(tmp_path))
    assert d["steps"] == steps and d["warmup"] == 3
    assert sorted(os.listdir(tmp_path)) == ["output0.npy"]
    got = np.load(tmp_path / "output0.npy")
    assert got.dtype == np.float32 and got.shape == (C, n)
    e = Engine(C, block=1024, max_samples=n)
    S.config3().apply(e)
    x = S.noise(C, n, seed=42)
    for _ in range(3 + steps):
        y = e.process(x)[0]
    assert_bit_exact(got, y, "dumped output vs the engine's last call")
