#!/usr/bin/env python
"""bench.py — channel-samples/s of the effect-node path on N B200s (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA engine
  python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU arithmetic (oracle port)
  python bench.py ... --dump-outputs DIR                   # also save the last timed step's outputs as .npy

A "step" is one dspb_process call over one batch of synthetic input: C channels x n samples per channel
(n = blocks_per_step device blocks), state carried across steps.  `value` is measured with inputs and outputs
resident in HBM; `e2e` goes through the host-buffer C-ABI call (pinned host memory, H2D and D2H inside the timed
region).

Scaling (SURVEY.md section 8e, north_star): the workload's channels are a FIXED total that is split over the ranks,
rank r of N owns channels [r*C/N, (r+1)*C/N) (`--scaling strong`, the default: "a 4096-channel chain on 8 B200").
`--scaling weak` gives every GPU the full channel count instead; with N > 1 the strong line also carries that figure as
`weak_scaling` so both readings come from one run.  Channels are independent: no data-path collective either way.

Besides the contract keys the line carries: `roofline` (dominant kernel, live CUDA-event timing), `parity_check` (a
channel subset of THIS configuration against the oracle, after the timed region), `sustained` (>= 2 s of back-to-back
steps with the clocks seen), `block_calls` (1024-sample calls, the BASELINE block size), `e2e`, `cpu_baseline`.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "channel_samples_per_sec"
UNIT = "channel-samples/s"
FIR_MODES = {0: "fft", 1: "direct_f64", 2: "toeplitz_tcgen05_bf16x2", 3: "fft_packed_f32x2"}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=os.environ.get("DSPB_BENCH_WORKLOAD", "target"))
    ap.add_argument("--scaling", default=os.environ.get("DSPB_BENCH_SCALING", "strong"), choices=["strong", "weak"])
    ap.add_argument("--channels", type=int, default=0,
                    help="strong: TOTAL channels over all GPUs; weak: channels per GPU (default: the workload's)")
    ap.add_argument("--block", type=int, default=1024, help="device block (samples)")
    ap.add_argument("--blocks-per-step", type=int, default=24,
                    help="device blocks per call; 24 x 1024 = 24576 samples = two 12288-sample FIR segments (one 16384-point window each)")
    ap.add_argument("--fir-mode", type=int, default=0)
    ap.add_argument("--iir-mode", type=int, default=0, help="1 = opt-in time-parallel recurrences where the measured error allows (not bit-exact)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline sample")
    ap.add_argument("--sustain-seconds", type=float, default=2.0, help="length of the sustained section (0 = skip)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-block-calls", action="store_true")
    ap.add_argument("--no-scan-side", action="store_true", help="skip the iir_mode=1 side measurement")
    ap.add_argument("--no-weak", action="store_true", help="skip the weak-scaling side measurement of a strong N>1 run")
    ap.add_argument("--gather", action="store_true", help="also time an NCCL gather of the outputs to rank 0")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write rank 0's outputs of the last timed step as DIR/output<i>.npy (float32), to compare two builds "
                         "(bench_outputs/ is ignored by git)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the CUDA engine's outputs: it needs --impl b200")
    return args


DEFAULT_CHANNELS = {"config1": 2, "config2": 256, "config2_one_pole": 256, "config3": 1024, "config4": 4096, "config5": 8192, "target": 4096}


def load_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of a kernel, from the committed `ncu --set full` captures:
    profiles/traffic.json, written by tools/ncu_traffic.py, keyed "workload/kind/channels/samples"."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(p))
    except Exception:
        return {}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def load_tensor_peak():
    """Dense bf16 TFLOP/s: the sustained figure (a kernel timed inside a long step), else the recipe's fallback."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["bf16_tflops_sustained"]), "measured sustained (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 1590.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while a timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return self

        def pump():
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])

        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()
        return self

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                pw.append(float(r[2]))
                for k, nm in enumerate(names):
                    if r[3 + k].lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "reasons": sorted(reasons), "samples": len(sm)}


def time_oracle(spec, channels, n, threads, steps=1, warmup=0):
    """Times the CPU oracle (the reference's arithmetic and 128-sample per-node block structure)."""
    from dsp_stuff_b200 import signals as S
    from oracle import oracle

    o = oracle.Oracle(channels, threads=threads)
    spec.apply(o)
    x = S.noise(channels, n)
    for _ in range(warmup):
        o.process(x)
    t0 = time.perf_counter()
    for _ in range(steps):
        o.process(x)
    dt = time.perf_counter() - t0
    return channels * n * steps / dt, dt


def cpu_baseline(spec, budget_s):
    cores = len(os.sched_getaffinity(0))
    # calibrate on a small sample, then size the real one to the budget
    n0 = 1024
    rate, dt = time_oracle(spec, cores, n0, cores)
    n = int(max(1024, min(48000 * 120, rate * budget_s / cores)) // 128 * 128)
    rate, dt = time_oracle(spec, cores, n, cores)
    # SURVEY §8d also asks for the single-thread figure: one channel, ~2 s
    r1, _ = time_oracle(spec, 1, n0, 1)
    n1 = int(max(1024, min(48000 * 60, r1 * 2.0)) // 128 * 128)
    r1, dt1 = time_oracle(spec, 1, n1, 1)
    return {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{cores} channels x {n} samples of the same graph and noise input, {cores} threads (one channel each), {dt:.1f} s",
            "single_thread": {"value": r1, "unit": UNIT, "cores": 1, "sample": f"1 channel x {n1} samples, {dt1:.1f} s"}}


def make_config(args, world, C_total, C_local, n):
    """The `config` object: identical for this repo's arm and the reference arm (same workload, same shape)."""
    return {"workload": args.workload, "scaling": args.scaling, "channels": C_total, "channels_per_gpu": C_local,
            "samples_per_step": n, "block": args.block, "blocks_per_step": args.blocks_per_step,
            "fir_mode": FIR_MODES[args.fir_mode], "iir_mode": {0: "exact", 1: "scan_where_probe_passes"}[args.iir_mode],
            "l2_policy": f"inputs+outputs {2 * C_local * n * 4 / 2**20:.0f} MiB per step per GPU"
                         + (" exceed the 126 MB L2" if 2 * C_local * n * 4 > 126e6 else " (smaller than the 126 MB L2: see weak_scaling / N=1 for the L2-exceeding size)")}


def shard_of(args, rank, world, C):
    """-> (first channel, local channel count, total channels of the job)"""
    from dsp_stuff_b200.shard import channel_range

    if args.scaling == "strong":
        lo, hi = channel_range(rank, world, C)
        return lo, hi - lo, C
    return rank * C, C, world * C


def run_reference(args, spec, C, n):
    """The reference's own CPU implementation of the path on the box's host cores: the oracle port (oracle/dsp_oracle.cpp;
    the Rust reference cannot be built in this image).  Each step is a bounded SAMPLE of the workload -- one channel per
    host core x ns samples -- and the figure is normalised per channel-sample, which is what the metric counts."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    _, C_local, C_total = shard_of(args, 0, max(1, world), C)
    cores = len(os.sched_getaffinity(0))
    rate0, _ = time_oracle(spec, cores, 1024, cores)
    # each step: a bounded sample (cores channels), sized so the whole run stays within ~2 minutes
    per_step = max(1.0, min(8.0, 100.0 / max(1, args.steps + args.warmup)))
    ns = int(max(1024, min(n, rate0 * per_step / cores)) // 128 * 128)
    rate, dt = time_oracle(spec, cores, ns, cores, steps=args.steps, warmup=args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": make_config(args, world, C_total, C_local, n),
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"each step = {cores} channels x {ns} samples of the workload graph (a bounded sample of the "
                                   f"{C_total} x {n} step, normalised per channel-sample; oracle/dsp_oracle.cpp = the reference's "
                                   f"arithmetic; the Rust reference cannot be built here), {cores} threads"},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


_REAL_STDOUT = None


def emit(line: dict):
    """The JSON line is the ONLY thing on stdout: libraries (NCCL prints its version banner there) were
    redirected to stderr at start-up."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is not None:
        os.write(_REAL_STDOUT, data)
    else:
        sys.stdout.write(data.decode())
        sys.stdout.flush()


def bind_host_side(local: int, world: int):
    """Best effort: run this rank's host threads (and first-touch its pinned buffers) on the NUMA node of its GPU, or,
    when the container shows a single node, on its own slice of the allowed cores so that N ranks do not share cores."""
    info = {"numa_node": None, "cpus": None}
    try:
        import torch

        allowed = sorted(os.sched_getaffinity(0))
        p = torch.cuda.get_device_properties(local)
        bdf = f"{getattr(p, 'pci_domain_id', 0):04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read().strip())
        cpus = []
        for part in open(f"/sys/bus/pci/devices/{bdf}/local_cpulist").read().strip().split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus += list(range(int(a), int(b) + 1))
            elif part:
                cpus.append(int(part))
        mine = [c for c in cpus if c in allowed]
        n_nodes = len([d for d in os.listdir("/sys/devices/system/node") if d.startswith("node")])
        info["numa_node"] = node
        info["numa_nodes_visible"] = n_nodes
        if node >= 0 and n_nodes > 1 and mine and len(mine) < len(allowed):
            os.sched_setaffinity(0, mine)
            info["cpus"] = f"{mine[0]}-{mine[-1]} ({len(mine)} cores, GPU-local NUMA node {node})"
        elif world > 1 and len(allowed) >= 2 * world:
            k = len(allowed) // world
            mine = allowed[local * k:(local + 1) * k]
            os.sched_setaffinity(0, mine)
            info["cpus"] = f"{mine[0]}-{mine[-1]} ({len(mine)} cores, one slice per rank)"
    except Exception as ex:  # noqa: BLE001
        info["error"] = str(ex)[:80]
    return info


def parity_check(args, spec, eng, x_dev, n, ch_offset):
    """A channel subset of the BENCHMARKED configuration (this engine, this size, device pointers, state carried over two
    calls) against the CPU oracle on the same seeded input.  FFT FIR => float-audio tolerance (1e-5 peak-relative and
    -100 dBFS rms); the warm-up samples and every graph without an FFT / libm node must match bit for bit."""
    import torch

    from dsp_stuff_b200 import signals as S
    from oracle import oracle

    C = eng.channels
    calls = 2
    sel = sorted({0, 1, C // 3, C // 2, C - 2, C - 1} & set(range(C)))
    eng.reset_state()
    n_out = eng._n_out
    ys = []
    for k in range(calls):
        # call k uses the same input block (what the timed loop feeds); the oracle gets the same sequence
        y = [torch.empty((C, n), dtype=torch.float32, device="cuda") for _ in range(n_out)]
        eng.process_device(x_dev, y, n)
        ys.append(y[0][sel].cpu().numpy())
    torch.cuda.synchronize()
    got = np.concatenate(ys, axis=1)
    o = oracle.Oracle(len(sel), threads=len(sel))
    spec.apply(o)
    xin = [np.ascontiguousarray(t[sel].cpu().numpy()) for t in x_dev]
    ref = np.concatenate([o.process(xin)[0] for _ in range(calls)], axis=1)
    d = got.astype(np.float64) - ref.astype(np.float64)
    peak = max(float(np.max(np.abs(ref))), 1e-30)
    rel = float(np.max(np.abs(d))) / peak
    rms = float(np.sqrt(np.mean(d * d)))
    dbfs = 20.0 * np.log10(rms) if rms > 0 else float("-inf")
    exact = bool(np.array_equal(got.view(np.uint32), ref.view(np.uint32)) or np.all((got == ref) | (np.isnan(got) & np.isnan(ref))))
    return {"channels": [int(c) + ch_offset for c in sel], "calls": calls, "samples_per_call": n, "rel": rel,
            "dbfs": None if dbfs == float("-inf") else float(dbfs), "bit_exact": exact,
            "pass": bool(exact or (rel <= 1e-5 and dbfs <= -100.0)), "tolerance": "1e-5 peak-relative and -100 dBFS rms (north_star)"}


DUMP_BYTES = 32 * 2**20


def dump_outputs(path, ys):
    """Writes the output arrays `ys` ([C, n] device tensors) as path/output<i>.npy.  When they exceed DUMP_BYTES in all,
    a fixed seeded sample of whole channels (the same rows of every output) is written instead, cut to fewer samples only
    if a single channel per output is already too large.  The bench input is seeded too, so equal arguments give files
    that two builds can be compared on."""
    import torch

    os.makedirs(path, exist_ok=True)
    C, n = ys[0].shape
    rows = max(1, min(C, DUMP_BYTES // (4 * n * len(ys))))
    cols = min(n, DUMP_BYTES // (4 * rows * len(ys)))
    sel = torch.from_numpy(np.sort(np.random.default_rng(0).choice(C, rows, replace=False))).to(ys[0].device)
    for i, y in enumerate(ys):
        np.save(os.path.join(path, f"output{i}.npy"), y.index_select(0, sel)[:, :cols].cpu().numpy())


def timed_steps(eng, x_dev, y_dev, n, steps, stream, barrier):
    import torch

    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(stream)
    for _ in range(steps):
        eng.process_device(x_dev, y_dev, n)
    ev1.record(stream)
    barrier()
    return ev0.elapsed_time(ev1)


def main():
    global _REAL_STDOUT
    args = parse_args()
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    from dsp_stuff_b200 import signals as S

    if args.workload not in S.WORKLOADS:
        raise SystemExit(f"unknown workload {args.workload}; have {sorted(S.WORKLOADS)}")
    factory, alg_bytes = S.WORKLOADS[args.workload]
    spec = factory()
    C = args.channels or DEFAULT_CHANNELS[args.workload]
    n = args.block * args.blocks_per_step

    if args.impl == "reference":
        run_reference(args, spec, C, n)
        return

    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback")
    torch.cuda.set_device(local)
    binding = bind_host_side(local, world)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    from dsp_stuff_b200.engine import Engine

    ch0, C_local, C_total = shard_of(args, rank, world, C)
    if C_local <= 0:
        raise SystemExit(f"rank {rank}: no channels to process ({C} channels over {world} ranks)")
    eng = Engine(C_local, block=args.block, max_samples=n, device=local, fir_mode=args.fir_mode, iir_mode=args.iir_mode)
    spec.apply(eng)
    n_in, n_out = eng._n_in, eng._n_out

    # synthetic input, identical on host and device; this rank's channels are [ch0, ch0 + C_local)
    x_host = [torch.from_numpy(S.noise(C_local, n, seed=42 + i, channel_offset=ch0)).pin_memory() for i in range(n_in)]
    y_host = [torch.empty((C_local, n), dtype=torch.float32).pin_memory() for _ in range(n_out)]
    x_dev = [t.cuda(non_blocking=True) for t in x_host]
    y_dev = [torch.empty((C_local, n), dtype=torch.float32, device="cuda") for _ in range(n_out)]
    stream = torch.cuda.current_stream()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(vals):
        t = torch.tensor(vals, dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t.tolist()]

    # ---- the contract's timed region: W warm-up steps, exactly K timed steps, device-resident ---------------------
    warm = max(3, args.warmup)
    for _ in range(warm):
        eng.process_device(x_dev, y_dev, n)
    launches_per_step = eng.kernel_launches
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    time.sleep(0.3)
    eng.profile(True)  # CUDA events around every kernel step, on the launching stream, inside the timed region
    ms = timed_steps(eng, x_dev, y_dev, n, args.steps, stream, barrier)
    clocks = sampler.stop() if rank == 0 else None
    step_times = eng.profile_read()
    eng.profile(False)
    plan = eng.plan_steps()
    (ms,) = allmax([ms])
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, y_dev)   # before any later section overwrites y_dev

    # ---- sustained: >= sustain_seconds of back-to-back steps (the 20-step figure is a burst at boost clocks) -------
    sustained = None
    if args.sustain_seconds > 0:
        per = max(ms / args.steps, 1e-3)
        chunk = max(args.steps, int(250.0 / per))  # ~0.25 s of steps between host synchronisations
        s2 = ClockSampler(local).start() if rank == 0 else None
        tot_ms, tot_steps = 0.0, 0
        t_start = time.perf_counter()
        while time.perf_counter() - t_start < args.sustain_seconds:
            tot_ms += timed_steps(eng, x_dev, y_dev, n, chunk, stream, barrier)
            tot_steps += chunk
            (go,) = allmax([1.0 if time.perf_counter() - t_start < args.sustain_seconds else 0.0])  # all ranks leave together
            if go == 0.0:
                break
        c2 = s2.stop() if s2 is not None else None
        (tot_ms,) = allmax([tot_ms])
        sustained = {"value": float(C_total) * n * tot_steps / (tot_ms * 1e-3), "unit": UNIT, "steps": tot_steps,
                     "seconds": tot_ms * 1e-3, "ms_per_step": tot_ms / tot_steps, "clocks": c2}

    # ---- 1024-sample calls: the BASELINE block size as the call size (launch-bound; the FIR window is 4x redundant) ---
    block_calls = None
    if not args.no_block_calls and n > args.block:
        xb = [t[:, :args.block].contiguous() for t in x_dev]
        yb = [torch.empty((C_local, args.block), dtype=torch.float32, device="cuda") for _ in range(n_out)]
        calls = max(50, args.steps * args.blocks_per_step)
        for _ in range(10):
            eng.process_device(xb, yb, args.block)
        bms = timed_steps(eng, xb, yb, args.block, calls, stream, barrier)
        (bms,) = allmax([bms])
        block_calls = {"samples_per_call": args.block, "calls": calls, "value": float(C_total) * args.block * calls / (bms * 1e-3),
                       "unit": UNIT, "ms_per_call": bms / calls, "launches_per_call": eng.kernel_launches}

    # ---- parity of the benchmarked configuration (rank 0's shard) -------------------------------------------------
    parity = None
    if not args.no_parity and rank == 0:
        try:
            parity = parity_check(args, spec, eng, x_dev, n, ch0)
        except Exception as ex:  # noqa: BLE001
            parity = {"pass": False, "error": str(ex)[:200]}
    barrier()

    # ---- end to end through the host-buffer C-ABI call (pinned memory; H2D + kernels + D2H per step) ---------------
    e2e_ms, e2e_sync_ms, h2d_ms, d2h_ms = 0.0, 0.0, 0.0, 0.0
    if not args.no_e2e:
        # (a) the blocking call, one step at a time
        for _ in range(2):
            eng.process_host(x_host, y_host, n)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            eng.process_host(x_host, y_host, n)
        torch.cuda.synchronize()
        e2e_sync_ms = (time.perf_counter() - t0) * 1e3
        # (b) the streaming form of the same call (DSPB_MEM_HOST_ASYNC + dspb_sync): two sets of pinned buffers, step k+1's
        # H2D runs next to step k's D2H; every step still copies its inputs in and its results out inside the timed region
        x_host2 = [t.clone().pin_memory() for t in x_host]
        y_host2 = [torch.empty_like(t).pin_memory() for t in y_host]
        sets = [(x_host, y_host), (x_host2, y_host2)]
        for k in range(2):
            eng.process_host(*sets[k % 2], n, wait=False)
        eng.sync()
        barrier()
        t0 = time.perf_counter()
        for k in range(args.steps):
            eng.process_host(*sets[k % 2], n, wait=False)
        eng.sync()
        e2e_ms = (time.perf_counter() - t0) * 1e3
        # the two copy directions alone, all ranks at once: what the host side (PCIe + host memory) gives this job
        reps = 5
        barrier()
        a0, a1, a2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        a0.record(stream)
        for _ in range(reps):
            for xh, xd in zip(x_host, x_dev):
                xd.copy_(xh, non_blocking=True)
        a1.record(stream)
        for _ in range(reps):
            for yh, yd in zip(y_host, y_dev):
                yh.copy_(yd, non_blocking=True)
        a2.record(stream)
        barrier()
        h2d_ms, d2h_ms = a0.elapsed_time(a1) / reps, a1.elapsed_time(a2) / reps

    gather_ms = None
    if args.gather and world > 1:
        outs = [torch.empty_like(y_dev[0]) for _ in range(world)] if rank == 0 else None
        dist.gather(y_dev[0], outs, dst=0)  # untimed: the first call sets up the NVLink connections
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record(stream)
        dist.gather(y_dev[0], outs, dst=0)
        g1.record(stream)
        barrier()
        gather_ms = g0.elapsed_time(g1)

    # ---- opt-in scan mode (iir_mode 1) next to the bit-exact default: same shard, same input ------------------------
    scan_side = None
    if args.iir_mode == 0 and not args.no_scan_side and any(nd.typename in ("biquad", "low_pass", "high_pass") for nd in spec.nodes):
        engs = Engine(C_local, block=args.block, max_samples=n, device=local, fir_mode=args.fir_mode, iir_mode=1)
        spec.apply(engs)
        verdicts = [ln.strip() for ln in engs.describe_plan().splitlines() if "scan" in ln and ("DF1(" in ln or "_pass(" in ln)]
        for _ in range(warm):
            engs.process_device(x_dev, y_dev, n)
        sms = timed_steps(engs, x_dev, y_dev, n, args.steps, stream, barrier)
        (sms,) = allmax([sms])
        sp = None
        if rank == 0 and not args.no_parity:
            try:
                sp = parity_check(args, spec, engs, x_dev, n, ch0)
            except Exception as ex:  # noqa: BLE001
                sp = {"pass": False, "error": str(ex)[:200]}
        barrier()
        scan_side = {"value": float(C_total) * n * args.steps / (sms * 1e-3), "unit": UNIT, "ms_per_step": sms / args.steps,
                     "iir_mode": "scan_where_probe_passes (opt-in, not bit-exact)", "filters": [v[:160] for v in verdicts],
                     "parity_check": sp}
        del engs

    # ---- weak-scaling side measurement of a strong run: every GPU takes the full channel count ---------------------
    weak = None
    if world > 1 and args.scaling == "strong" and not args.no_weak:
        del eng
        xw = [torch.from_numpy(S.noise(C, n, seed=42 + i, channel_offset=rank * C)).cuda() for i in range(n_in)]
        yw = [torch.empty((C, n), dtype=torch.float32, device="cuda") for _ in range(n_out)]
        engw = Engine(C, block=args.block, max_samples=n, device=local, fir_mode=args.fir_mode, iir_mode=args.iir_mode)
        spec.apply(engw)
        for _ in range(warm):
            engw.process_device(xw, yw, n)
        wms = timed_steps(engw, xw, yw, n, args.steps, stream, barrier)
        (wms,) = allmax([wms])
        weak = {"value": float(world) * C * n * args.steps / (wms * 1e-3), "unit": UNIT, "channels_per_gpu": C,
                "ms_per_step": wms / args.steps, "scaling": "weak"}

    e2e_ms, e2e_sync_ms, gather_ms, h2d_ms, d2h_ms = allmax([e2e_ms, e2e_sync_ms, gather_ms or 0.0, h2d_ms, d2h_ms])

    if rank == 0:
        total = float(C_total) * n * args.steps
        value = total / (ms * 1e-3)
        peak, peak_src = load_peaks()
        traffic = load_traffic()
        # dominant kernel = the schedule step with the largest summed device time; its achieved bandwidth is
        # its own ALGORITHMIC bytes per launch (per channel-sample figure x C x n) / its average launch time
        kernels = []
        for i, (tot_ms, rounds) in enumerate(step_times):
            if rounds:
                avg = tot_ms / rounds
                kernels.append({"step": i, "kind": plan[i]["kind"], "alg_bytes_per_channel_sample": plan[i]["alg_bytes"],
                                "avg_ms": avg, "share_of_step": tot_ms / ms,
                                "achieved_gbs": plan[i]["alg_bytes"] * C_local * n / (avg * 1e-3) / 1e9})
        dom = max(kernels, key=lambda k: k["avg_ms"])
        per_gpu_rate = C_local * n * args.steps / (ms * 1e-3)
        achieved = dom["achieved_gbs"]
        step_achieved = alg_bytes * per_gpu_rate / 1e9
        cfg = make_config(args, world, C_total, C_local, n)
        cfg["x_realtime_per_channel"] = value / C_total / 48000.0
        if binding.get("cpus"):
            cfg["host_binding"] = binding["cpus"]
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": cfg,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic.get(f"{args.workload}/{dom['kind']}/{C_local}/{n}"), "peak_source": peak_src,
                         "kernel": f"step {dom['step']} ({dom['kind']})", "kernel_avg_ms": dom["avg_ms"],
                         "kernel_alg_bytes_per_channel_sample": dom["alg_bytes_per_channel_sample"],
                         "kernel_share_of_step": dom["share_of_step"], "kernels": kernels,
                         "whole_step": {"alg_bytes_per_channel_sample": alg_bytes, "achieved": step_achieved,
                                        "frac": step_achieved / peak, "frac_of_8000_nominal": step_achieved / 8000.0}},
            "gpu_launches": int(launches_per_step * args.steps),
            "clocks": clocks,
        }
        if args.fir_mode == 2 and dom["kind"] == "fir":
            # Toeplitz tensor-core FIR: the bounding roofline is the tensor pipe.  Algorithmic flops of the kernel =
            # 3 split-bf16 products x 2 N flop per channel-sample (N taps), all launches of the step (split pre-pass included)
            n_taps = max([len(nd.taps) for nd in spec.nodes if nd.typename == "fir" and nd.taps is not None] or [1])
            tf = 3 * 2 * n_taps * C_local * n / (dom["avg_ms"] * 1e-3) / 1e12
            tpeak, tsrc = load_tensor_peak()
            line["roofline"].update({"bound": "tensor", "achieved": tf, "peak": tpeak, "unit": "TFLOP/s", "frac": tf / tpeak,
                                     "peak_source": tsrc, "traffic": None,
                                     "flops_per_channel_sample": 3 * 2 * n_taps,
                                     "hbm_view": {"achieved_gbs": achieved, "peak_gbs": peak}})
        if sustained:
            line["sustained"] = sustained
        if block_calls:
            line["block_calls"] = block_calls
        if parity is not None:
            line["parity_check"] = parity
        if scan_side:
            line["scan_mode"] = scan_side
        if weak:
            line["weak_scaling"] = weak
        if not args.no_e2e:
            bi, bo = n_in * C_local * n * 4, n_out * C_local * n * 4
            line["e2e"] = {"value": float(C_total) * n * args.steps / (e2e_ms * 1e-3), "unit": UNIT,
                           "h2d_bytes_per_step": bi, "d2h_bytes_per_step": bo, "ms_per_step": e2e_ms / args.steps,
                           "api": "dspb_process(DSPB_MEM_HOST_ASYNC) per step on alternating pinned buffer sets + dspb_sync",
                           "blocking_call": {"value": float(C_total) * n * args.steps / (e2e_sync_ms * 1e-3), "unit": UNIT,
                                             "ms_per_step": e2e_sync_ms / args.steps, "api": "dspb_process(DSPB_MEM_HOST), returns when the outputs are complete"},
                           "copies_alone": {"h2d_ms": h2d_ms, "d2h_ms": d2h_ms,
                                            "h2d_gbs_per_gpu": bi / (h2d_ms * 1e-3) / 1e9 if h2d_ms else None,
                                            "d2h_gbs_per_gpu": bo / (d2h_ms * 1e-3) / 1e9 if d2h_ms else None,
                                            "note": "the two directions alone, all ranks copying at once (max over ranks): the host-side bound of e2e"}}
        if gather_ms:
            line["gather_to_rank0_ms"] = gather_ms
        if not args.no_cpu_baseline and world == 1:   # rank 0 at N = 1 only; at N > 1 this rank is pinned to its core slice
            line["cpu_baseline"] = cpu_baseline(spec, args.cpu_seconds)
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
