"""Cost of per-channel parameters (Engine.set_f32_channels) on the GPU.

Target chain (gain -> distort(SoftClip) -> biquad -> reverb -> FIR 4096, FFT FIR), 4096 channels x 24576 samples per step,
device pointers.  Three arms in one process, alternated round by round, each timed with CUDA events for at least
--seconds per round:
  shared     every parameter shared (the compiled ChainGDBR kernel)
  pc_equal   per-channel calls with all values equal (collapse to the shared case: same plan, same kernels)
  pc_dist    distinct values per channel: gain.level, distort.level, reverb.decay and RBJ low-pass biquad coefficients with
             the cutoff spread over 500 Hz - 4 kHz (the interpreter, ChainDynamic, in the same warp-specialised kernel)
Then config2 (biquad -> biquad, the two-recurrence kernel) at 256 channels, shared vs per-channel coefficients.
Prints channel-samples/s per arm, the per-step split from dspb_profile_*, and the GPU name and power limit.

    python tools/per_channel_bench.py [--seconds 2] [--rounds 3]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from dsp_stuff_b200 import signals as S  # noqa: E402
from dsp_stuff_b200.engine import FIR_DIRECT, FIR_FFT, Engine  # noqa: E402


def gpu_info():
    import torch

    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = q
    except Exception as ex:  # noqa: BLE001
        info["power_limit_and_max_sm_clock"] = f"unavailable ({ex})"
    return info


def spread(vals, C, k=0):
    vals = np.asarray(vals, dtype=np.float32)
    return vals[(np.arange(C) * (2 * k + 1) + k) % len(vals)]


def build(graph, C, T, fir_mode, arm, pc_fields):
    e = Engine(C, block=128, max_samples=T, fir_mode=fir_mode)
    graph.apply(e)
    if arm == "pc_equal":
        for nd in graph.nodes:
            for f, v in nd.f32.items():
                if (nd.id, f) in pc_fields:
                    e.set_f32_channels(nd.id, f, np.full(C, v, dtype=np.float32))
    elif arm == "pc_dist":
        for (nid, f), v in pc_fields.items():
            e.set_f32_channels(nid, f, v)
    return e


def time_arm(e, x, y, T, seconds):
    import torch

    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e.process_device([x], [y], T)   # lowering / table upload outside the window
    torch.cuda.synchronize()
    steps, ms = 0, 0.0
    while ms < seconds * 1000.0:
        ev0.record()
        for _ in range(4):
            e.process_device([x], [y], T)
        ev1.record()
        ev1.synchronize()
        ms += ev0.elapsed_time(ev1)
        steps += 4
    return steps, ms


def profile(e, x, y, T, reps=8):
    import torch

    e.profile(True)
    for _ in range(reps):
        e.process_device([x], [y], T)
    torch.cuda.synchronize()
    e.profile(False)
    kinds = [s["kind"] for s in e.plan_steps()]
    return [{"step": i, "kind": kinds[i] if i < len(kinds) else "?", "ms": ms / max(r, 1)} for i, (ms, r) in enumerate(e.profile_read())]


def run_workload(name, graph, C, T, fir_mode, pc_fields, seconds, rounds):
    import torch

    x = torch.from_numpy(S.noise(C, T)).cuda()
    y = torch.empty((C, T), dtype=torch.float32, device="cuda")
    arms = ["shared", "pc_equal", "pc_dist"]
    engines = {a: build(graph, C, T, fir_mode, a, pc_fields) for a in arms}
    acc = {a: [0, 0.0] for a in arms}
    for _ in range(rounds):
        for a in arms:
            s, ms = time_arm(engines[a], x, y, T, seconds)
            acc[a][0] += s
            acc[a][1] += ms
    out = {"workload": name, "channels": C, "samples_per_step": T, "arms": {}}
    for a in arms:
        steps, ms = acc[a]
        out["arms"][a] = {"ms_per_step": ms / steps, "channel_samples_per_s": C * T * steps / (ms / 1000.0),
                          "steps": steps, "profile": profile(engines[a], x, y, T),
                          "launches": engines[a].kernel_launches}
    base = out["arms"]["shared"]["ms_per_step"]
    for a in arms:
        out["arms"][a]["vs_shared"] = out["arms"][a]["ms_per_step"] / base
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=2.0, help="timed seconds per arm and round")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None, help="write the JSON here as well")
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement needs the GPU")
    C = 4096
    lp = [S.rbj_biquad("lp", f) for f in np.linspace(500.0, 4000.0, 64)]
    pc_target = {(0, "level"): spread(np.linspace(0.5, 3.0, 64), C, 1), (1, "level"): spread(np.linspace(1.0, 6.0, 64), C, 2),
                 (3, "decay"): spread(np.linspace(0.2, 0.8, 64), C, 3)}
    for k in ("a1", "a2", "b0", "b1", "b2"):
        pc_target[(2, k)] = spread([r[k] for r in lp], C)
    res = {"gpu": gpu_info(), "results": []}
    res["results"].append(run_workload("target", S.target_chain(4096), C, 24576, FIR_FFT, pc_target, a.seconds, a.rounds))
    C2 = 256
    hp = [S.rbj_biquad("hp", f) for f in np.linspace(100.0, 800.0, 64)]
    pc2 = {}
    for k in ("a1", "a2", "b0", "b1", "b2"):
        pc2[(0, k)] = spread([r[k] for r in lp], C2)
        pc2[(1, k)] = spread([r[k] for r in hp], C2, 1)
    res["results"].append(run_workload("config2", S.config2(), C2, 24576, FIR_DIRECT, pc2, a.seconds, a.rounds))
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
