"""Cost of per-channel state resets (Engine.reset_channels) on the GPU.

Workloads, 4096 channels, target chain (gain -> distort -> biquad -> reverb -> FFT FIR with 4096 taps), device pointers:
  target         24576 samples per call (wide + narrow segment kernels)
  target_1024    1024 samples per call (the UPC kernel: a reset re-primes its delay line)
Arms, alternated round by round in one process, each timed for at least --seconds per round; the reset is recorded before
every call, so every call pays the clear and the warm-up patch of the channels reset just before it:
  none           no reset
  reset1         channel 2049
  reset64        64 scattered channels (every 64th, starting at 17)
  reset4096      every channel
  reset_state    dspb_reset_state before every call (synchronises the device)
Whole-call time from CUDA events around the calls; the fused and FIR step times from dspb_profile_* (the clear launch is
outside every step: whole call minus the steps).
Streaming: the asynchronous host path (DSPB_MEM_HOST_ASYNC, pinned buffers, 4096 x 1024) with one reset every call against
none, host wall clock over the calls: the upload / download overlap must survive.
Prints the GPU name and power limit.

    python tools/reset_channels_bench.py [--seconds 2] [--rounds 3] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from dsp_stuff_b200 import signals as S  # noqa: E402
from dsp_stuff_b200.engine import FIR_FFT, Engine  # noqa: E402

C, N = 4096, 4096
ARMS = {
    "none": None,
    "reset1": np.array([2049], dtype=np.int32),
    "reset64": np.arange(17, C, 64, dtype=np.int32),
    "reset4096": np.arange(C, dtype=np.int32),
    "reset_state": "state",
}


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


def build(T):
    e = Engine(C, block=128, max_samples=T, fir_mode=FIR_FFT)
    S.target_chain(N).apply(e)
    return e


def before_call(e, arm):
    if isinstance(arm, str):
        e.reset_state()
    elif arm is not None:
        e.reset_channels(arm)


def time_arm(e, arm, x, y, T, seconds):
    """-> (calls, ms of whole calls, ms of the fused steps, ms of the FIR steps) over at least `seconds`."""
    import torch

    kinds = [s["kind"] for s in e.plan_steps()]
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    calls, ms, step_ms = 0, 0.0, {"fused": 0.0, "fir": 0.0}
    while ms < seconds * 1000.0:
        e.profile(True)
        ev0.record()
        for _ in range(8):
            before_call(e, arm)
            e.process_device([x], [y], T)
        ev1.record()
        ev1.synchronize()
        e.profile(False)
        for i, (t, r) in enumerate(e.profile_read()):
            step_ms[kinds[i]] += t / max(r, 1) * 8
        ms += ev0.elapsed_time(ev1)
        calls += 8
    return calls, ms, step_ms["fused"], step_ms["fir"]


def run_workload(name, T, seconds, rounds):
    import torch

    x = torch.from_numpy(S.noise(C, T)).cuda()
    y = torch.empty((C, T), dtype=torch.float32, device="cuda")
    engines = {a: build(T) for a in ARMS}
    for a, e in engines.items():   # lowering, spectra and the first launches outside the timed window
        for _ in range(2):
            before_call(e, ARMS[a])
            e.process_device([x], [y], T)
    torch.cuda.synchronize()
    acc = {a: np.zeros(4) for a in ARMS}
    for _ in range(rounds):
        for a, e in engines.items():
            acc[a] += time_arm(e, ARMS[a], x, y, T, seconds)
    out = {"workload": name, "channels": C, "samples_per_call": T, "n_taps": N, "arms": {}}
    for a in ARMS:
        calls, ms, fused, fir = acc[a]
        out["arms"][a] = {"ms_per_call": ms / calls, "fused_ms": fused / calls, "fir_ms": fir / calls,
                          "outside_steps_ms": (ms - fused - fir) / calls, "calls": int(calls)}
    del engines
    torch.cuda.synchronize()
    return out


def run_streaming(seconds, rounds, T=1024):
    import torch

    xs = [torch.from_numpy(S.noise(C, T, sample_offset=k * T)).pin_memory() for k in range(2)]
    ys = [torch.empty((C, T), dtype=torch.float32).pin_memory() for _ in range(2)]
    arms = {"none": None, "reset1_every_call": np.array([2049], dtype=np.int32)}
    engines = {a: build(T) for a in arms}
    for e in engines.values():
        e.process_host([xs[0]], [ys[0]], T)
    acc = {a: [0, 0.0] for a in arms}
    for _ in range(rounds):
        for a, e in engines.items():
            calls, t0 = 0, time.perf_counter()
            while time.perf_counter() - t0 < seconds:
                for k in range(16):
                    before_call(e, arms[a])
                    e.process_host([xs[k % 2]], [ys[k % 2]], T, wait=False)   # two buffer pairs in flight
                calls += 16
            e.sync()
            acc[a][0] += calls
            acc[a][1] += (time.perf_counter() - t0) * 1000.0
    return {"workload": "streaming_host_async", "channels": C, "samples_per_call": T,
            "arms": {a: {"ms_per_call": ms / calls, "calls": calls,
                         "channel_samples_per_s": C * T * calls / (ms / 1000.0)} for a, (calls, ms) in acc.items()}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=2.0, help="timed seconds per arm and round")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None, help="write the JSON here as well")
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement needs the GPU")
    res = {"gpu": gpu_info(), "results": []}
    for name, T in [("target", 24576), ("target_1024", 1024)]:
        r = run_workload(name, T, a.seconds, a.rounds)
        res["results"].append(r)
        print(json.dumps({"workload": name} | {arm: round(v["ms_per_call"], 4) for arm, v in r["arms"].items()}), flush=True)
    r = run_streaming(a.seconds, a.rounds)
    res["results"].append(r)
    print(json.dumps({"workload": r["workload"]} | {arm: round(v["ms_per_call"], 4) for arm, v in r["arms"].items()}), flush=True)
    res["gpu_after"] = gpu_info()
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
