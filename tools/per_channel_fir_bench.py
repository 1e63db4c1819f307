"""Cost of per-channel FIR impulse responses (Engine.set_taps_channels) on the GPU.

Workloads, 4096 channels, FFT FIR with 4096 taps, device pointers:
  config4        input -> fir -> output, 24576 samples per call (wide + narrow segment kernels)
  target         gain -> distort -> biquad -> reverb -> fir, 24576 samples per call
  config4_1024   config4 with 1024-sample calls (the UPC kernel)
Arms, alternated round by round in one process, each timed for at least --seconds per round:
  shared         set_taps: one impulse response
  pc_equal       set_taps_channels with 8 identical rows (collapses to shared: same plan and kernels)
  bank8_inter    8 impulse responses, channel c uses c % 8 (4 channels per set in every 32-channel group: no single transforms)
  bank8_runs     8 impulse responses in contiguous runs of 512 channels
  distinct       4096 impulse responses, one per channel (one channel per transform)
The FIR step time comes from dspb_profile_* (CUDA events around each step); the whole step from events around the calls.
Prints the H-table (spectra) memory per arm and the GPU name and power limit.

    python tools/per_channel_fir_bench.py [--seconds 2] [--rounds 3] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from dsp_stuff_b200 import signals as S  # noqa: E402
from dsp_stuff_b200.engine import FIR_FFT, Engine  # noqa: E402

ARMS = ["shared", "pc_equal", "bank8_inter", "bank8_runs", "distinct"]
SPECTRUM_KIB = 320   # fir_fft_spectrum_bytes() of one tap set


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


def irs(K, N, seed=0):
    rng = np.random.default_rng(seed)
    env = np.exp(-np.arange(N) / (N / 4.0 + 1.0))
    return (rng.standard_normal((K, N)) * env * 0.1)[:, ::-1].copy()


def build(graph, fir_node, C, T, N, arm):
    e = Engine(C, block=128, max_samples=T, fir_mode=FIR_FFT)
    graph.apply(e)
    c = np.arange(C, dtype=np.int32)
    if arm == "shared":
        e.set_taps(fir_node, irs(1, N)[0])
    elif arm == "pc_equal":
        e.set_taps_channels(fir_node, np.repeat(irs(1, N), 8, axis=0), c % 8)
    elif arm == "bank8_inter":
        e.set_taps_channels(fir_node, irs(8, N), c % 8)
    elif arm == "bank8_runs":
        e.set_taps_channels(fir_node, irs(8, N), c * 8 // C)
    else:
        e.set_taps_channels(fir_node, irs(C, N), c)
    return e


def fir_listing(e):
    line = next(s["text"] for s in e.plan_steps() if s["kind"] == "fir")
    m = re.search(r"per-channel taps: (\d+) sets, (\d+) transforms \((\d+) single", line)
    return (1, None, None) if m is None else tuple(int(g) for g in m.groups())


def time_arm(e, x, y, T, seconds):
    """-> (steps, ms of whole steps, ms of the FIR step) over at least `seconds`."""
    import torch

    fir_idx = [i for i, s in enumerate(e.plan_steps()) if s["kind"] == "fir"]
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    steps, ms, fir_ms, fir_rounds = 0, 0.0, 0.0, 0
    while ms < seconds * 1000.0:
        e.profile(True)
        ev0.record()
        for _ in range(8):
            e.process_device([x], [y], T)
        ev1.record()
        ev1.synchronize()
        e.profile(False)
        prof = e.profile_read()
        for i in fir_idx:
            fir_ms += prof[i][0]
            fir_rounds += prof[i][1]
        ms += ev0.elapsed_time(ev1)
        steps += 8
    return steps, ms, fir_ms / max(fir_rounds, 1) * steps


def run_workload(name, graph, fir_node, C, T, N, seconds, rounds):
    import torch

    x = torch.from_numpy(S.noise(C, T)).cuda()
    y = torch.empty((C, T), dtype=torch.float32, device="cuda")
    engines = {a: build(graph, fir_node, C, T, N, a) for a in ARMS}
    for e in engines.values():   # lowering, spectra and the first launches outside the timed window
        e.process_device([x], [y], T)
        e.process_device([x], [y], T)
    torch.cuda.synchronize()
    acc = {a: [0, 0.0, 0.0] for a in ARMS}
    for _ in range(rounds):
        for a in ARMS:
            s, ms, fms = time_arm(engines[a], x, y, T, seconds)
            acc[a][0] += s
            acc[a][1] += ms
            acc[a][2] += fms
    out = {"workload": name, "channels": C, "samples_per_call": T, "n_taps": N, "arms": {}}
    for a in ARMS:
        steps, ms, fms = acc[a]
        K, xf, single = fir_listing(engines[a])
        out["arms"][a] = {"ms_per_step": ms / steps, "fir_ms_per_step": fms / steps, "steps": steps, "sets": K,
                          "transforms": xf if xf is not None else (C + 1) // 2, "single_channel": single or 0,
                          "h_table_mib": K * SPECTRUM_KIB / 1024.0}
    base = out["arms"]["shared"]["fir_ms_per_step"]
    for a in ARMS:
        out["arms"][a]["fir_vs_shared"] = out["arms"][a]["fir_ms_per_step"] / base
    del engines
    torch.cuda.synchronize()
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
    C, N = 4096, 4096
    res = {"gpu": gpu_info(), "results": []}
    for name, graph, node, T in [("config4", S.config4(N), 0, 24576), ("target", S.target_chain(N), 4, 24576),
                                 ("config4_1024", S.config4(N), 0, 1024)]:
        r = run_workload(name, graph, node, C, T, N, a.seconds, a.rounds)
        res["results"].append(r)
        print(json.dumps({k: r[k] for k in ("workload", "samples_per_call")} |
                         {arm: (round(v["fir_ms_per_step"], 4), round(v["ms_per_step"], 4)) for arm, v in r["arms"].items()}),
              flush=True)
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
