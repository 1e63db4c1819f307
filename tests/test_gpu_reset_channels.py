"""Per-channel state reset (dspb_reset_channels) on the GPU.

Reference: every channel's output comes from the CPU oracle it was last started on.  At first one oracle runs all channels;
a reset starts a fresh oracle over just the reset channels (grouped by their per-channel settings), fed only the input after
the reset, while every other channel keeps its continuing oracle.  Graphs without an FFT / Toeplitz FIR and fir_mode 1 must be
bit-exact; with the FFT or Toeplitz FIR the warm-up samples (the first N - 1 since a channel's reset, recomputed by the direct
kernel) must be bit-exact and the rest within the parity tolerance, each oracle's channels against their own level.

Isolation: channels that were not reset must equal a twin engine that never reset (bit for bit, except next to the FFT FIR,
where two channels share one complex transform and a zeroed partner history changes the rounding).
"""
import numpy as np
import pytest

from dsp_stuff_b200 import GraphSpec
from dsp_stuff_b200 import signals as S
from tests.util import assert_audio_close, assert_bit_exact, make_oracle

pytestmark = pytest.mark.gpu
FIR_FFT, FIR_DIRECT, FIR_TOEPLITZ = 0, 1, 2
C = 70                              # not a multiple of 32: a partial last CTA group and launch range
R1 = [0, 69, 31, 32, 31, 0]         # first and last channel, both sides of 31/32, channel 32 of the FFT pair (32, 33), duplicates
R2 = [5, 40, 41, 69]
R3 = [0, 33, 64, 65, 66, 67, 68]


class Ref:
    """Oracles that follow an engine through per-channel resets.  key(c) groups channels that need differently configured
    oracles (per-channel settings); setup(oracle, key) configures one."""

    def __init__(self, oracle_mod, spec, C, key=None, setup=None, ring_granule=1024):
        self.mod, self.spec, self.C, self.granule = oracle_mod, spec, C, ring_granule
        self.key = key or (lambda c: ())
        self.setup = setup or (lambda o, k: None)
        self.parts = []                                  # [channels, oracle, still-owned mask]
        self.since = np.zeros(C, dtype=np.int64)         # samples each channel's oracle has seen
        self.start(range(C))

    def start(self, channels):
        chans = sorted(set(int(c) for c in channels))
        for p in self.parts:
            p[2] &= ~np.isin(p[0], chans)
        keys = {c: self.key(c) for c in chans}
        for k in dict.fromkeys(keys.values()):
            sel = np.array([c for c in chans if keys[c] == k])
            o = make_oracle(self.mod, self.spec, len(sel), ring_granule=self.granule)
            self.setup(o, k)
            self.parts.append([sel, o, np.ones(len(sel), dtype=bool)])
        self.since[chans] = 0

    def set_taps(self, node, taps):                      # set_taps clears every channel's history, like the engine's
        for _, o, _ in self.parts:
            o.set_taps(node, taps)
        self.since[:] = 0

    def groups(self):
        return [p[0][p[2]] for p in self.parts if p[2].any()]

    def process(self, x, n):
        out = np.zeros((self.C, n), dtype=np.float32)
        self.parts = [p for p in self.parts if p[2].any()]
        for sel, o, own in self.parts:
            y = o.process([np.ascontiguousarray(x[sel])])[0] if x is not None else o.process_n(n)[0]
            out[sel[own]] = y[own]
        return out


def engine(spec, C, n, fir_mode=FIR_FFT, **kw):
    from dsp_stuff_b200.engine import Engine

    e = Engine(C, block=128, max_samples=n, fir_mode=fir_mode, **kw)
    spec.apply(e)
    return e


def check(got, want, ref, since, N, exact, what):
    """got / want: one call; since: samples each channel's oracle had seen before it."""
    if exact:
        assert_bit_exact(got, want, what)
        return
    for c in range(got.shape[0]):
        warm = max(0, min(got.shape[1], N - 1 - int(since[c])))
        if warm:
            assert_bit_exact(got[c, :warm], want[c, :warm], f"{what} channel {c} warm-up")
    for g in ref.groups():
        assert_audio_close(got[g], want[g], what=f"{what} channels {g[:4]}...")


def run(e, ref, calls, resets, N=1, exact=True, twin=None, twin_exact=True, seed=0, has_input=True, what=""):
    """calls[k] samples per call; resets[k] (if any) is reset on the engine and the reference before call k."""
    t = 0
    for k, n in enumerate(calls):
        if k in resets:
            e.reset_channels(resets[k])
            ref.start(resets[k])
        x = S.noise(e.channels, n, seed=seed, sample_offset=t) if has_input else None
        since = ref.since.copy()
        got = e.process([x] if has_input else [], n)[0]
        want = ref.process(x, n)
        ref.since += n
        check(got, want, ref, since, N, exact, f"{what} call {k} (n={n})")
        if twin is not None:
            other = twin.process([x] if has_input else [], n)[0]
            keep = np.flatnonzero(ref.since == np.max(ref.since))       # channels never reset
            if twin_exact:
                assert_bit_exact(got[keep], other[keep], f"{what} call {k}: unreset channels vs twin")
            else:
                assert_audio_close(got[keep], other[keep], what=f"{what} call {k}: unreset channels vs twin")
        t += n


def chain(typename, **params):
    g = GraphSpec().node(10, "input").node(0, typename, **params).node(11, "output")
    return g.link(10, "out", 0, "in").link(0, "out", 11, "in")


NODE_GRAPHS = {
    "biquad": (chain("biquad", **S.rbj_biquad("lp", 1000.0)), 1024),
    "low_pass": (chain("low_pass", ratio=0.9), 1024),
    "high_pass": (chain("high_pass", ratio=0.99), 1024),
    "envelope": (chain("envelope", attack=20.0, release=400.0), 1024),
    "gate": (chain("gate", threshold=0.3, attack=5.0, release=200.0), 1024),
    "reverb": (chain("reverb", seconds=0.25, decay=0.5), 1024),
    "reverb_granule1": (chain("reverb", seconds=0.01021, decay=0.7), 1),   # D = 490: rows not 16-byte aligned
    "config3": (S.config3(), 1024),
}
CALLS = [1024, 128 * 7, 2048, 128 * 88]
RESETS = {1: R1, 2: R2, 3: R3}


@pytest.mark.parametrize("name", list(NODE_GRAPHS))
def test_stateful_node_bit_exact_and_isolated(oracle_mod, name):
    spec, granule = NODE_GRAPHS[name]
    e, twin = engine(spec, C, max(CALLS), ring_granule=granule), engine(spec, C, max(CALLS), ring_granule=granule)
    ref = Ref(oracle_mod, spec, C, ring_granule=granule)
    run(e, ref, CALLS, RESETS, twin=twin, what=name)


@pytest.mark.parametrize("mode,exact", [("Triangle", True), ("Square", True), ("Constant", True), ("Sine", False)])
def test_signal_gen_restarts_its_clock(oracle_mod, mode, exact):
    g = GraphSpec().node(0, "signal_gen", mode=mode, amplitude=0.5, frequency=997.0).node(1, "gain", level=1.5).node(11, "output")
    g.link(0, "out", 1, "in").link(1, "out", 11, "in")
    e, twin = engine(g, C, max(CALLS)), engine(g, C, max(CALLS))
    ref = Ref(oracle_mod, g, C)
    run(e, ref, CALLS, RESETS, exact=exact, N=1, twin=twin, has_input=False, what=f"signal_gen {mode}")


@pytest.mark.parametrize("fir_mode", [FIR_FFT, FIR_DIRECT, FIR_TOEPLITZ])
def test_target_chain_every_fir_mode(oracle_mod, fir_mode):
    N = 300
    spec = S.target_chain(N)
    calls = [2048, 1024, 128 * 88, 4096, 1024]
    e, twin = engine(spec, C, max(calls), fir_mode), engine(spec, C, max(calls), fir_mode)
    ref = Ref(oracle_mod, spec, C)
    exact = fir_mode == FIR_DIRECT
    run(e, ref, calls, {1: R1, 3: R2, 4: R3}, N=N, exact=exact, twin=twin, twin_exact=exact, what=f"fir_mode {fir_mode}")


def test_warm_up_across_calls_upc_and_ragged_segments(oracle_mod):
    """4096 taps: 1024-sample calls (UPC kernel, re-primed after each reset) and ragged 128 * 88 segment calls.  The first
    reset comes while the whole engine is still in its warm-up, the second restarts channels in the middle of their own."""
    N = 4096
    spec = S.config4(N)
    calls = [1024, 1024, 1024, 1024, 1024, 128 * 88, 1024, 128 * 88, 1024, 1024]
    resets = {1: R1, 3: [0, 31, 5], 5: R2, 6: R3, 8: [69]}
    e, twin = engine(spec, C, max(calls)), engine(spec, C, max(calls))
    ref = Ref(oracle_mod, spec, C)
    run(e, ref, calls, resets, N=N, exact=False, twin=twin, twin_exact=False, what="4096 taps")


def test_warm_up_across_calls_direct_mode_bit_exact(oracle_mod):
    N = 1500
    spec = S.config4(N)
    calls = [512, 512, 128 * 3, 512, 128 * 5, 2048]
    e = engine(spec, C, max(calls), FIR_DIRECT)
    ref = Ref(oracle_mod, spec, C)
    run(e, ref, calls, {1: R1, 2: [0, 40], 4: R2}, N=N, exact=True, what="direct")


def test_reset_then_set_taps(oracle_mod):
    N = 300
    spec = S.config4(N)
    e = engine(spec, C, 4096)
    ref = Ref(oracle_mod, spec, C)
    run(e, ref, [2048], {}, N=N, exact=False)
    e.reset_channels(R1)
    ref.start(R1)
    new = S.reverb_ir(N, seed=3)[::-1].copy()
    e.set_taps(0, new)
    ref.set_taps(0, new)
    t = 2048
    for k, n in enumerate([1024, 128 * 10, 4096]):
        x = S.noise(C, n, sample_offset=t)
        since = ref.since.copy()
        got = e.process([x])[0]
        want = ref.process(x, n)
        ref.since += n
        check(got, want, ref, since, N, False, f"after set_taps call {k}")
        t += n


@pytest.mark.parametrize("kind", ["bank8", "distinct"])
def test_per_channel_settings_survive_a_reset(oracle_mod, kind):
    N, FIR = 300, 4
    spec = S.target_chain(N)
    rng = np.random.default_rng(1)
    env = np.exp(-np.arange(N) / (N / 4.0 + 1.0))
    K = 8 if kind == "bank8" else C
    bank = (rng.standard_normal((K, N)) * env * 0.1)[:, ::-1].copy()
    idx = (np.arange(C) % K).astype(np.int32)
    level = np.array([0.5, 1.0, 2.0], dtype=np.float32)[np.arange(C) % 3]
    e = engine(spec, C, 4096)
    e.set_taps_channels(FIR, bank, idx)
    e.set_f32_channels(0, "level", level)

    def setup(o, k):
        o.set_taps(FIR, bank[k[0]])
        o.set_f32(0, "level", k[1])

    ref = Ref(oracle_mod, spec, C, key=lambda c: (int(idx[c]), float(level[c])), setup=setup)
    run(e, ref, [2048, 1024, 4096, 1024], {1: R1, 3: R2}, N=N, exact=False, what=kind)


@pytest.mark.parametrize("spec_name", ["config3", "target"])
def test_resetting_every_channel_equals_reset_state(spec_name):
    spec = S.config3() if spec_name == "config3" else S.target_chain(300)
    a, b = engine(spec, C, 4096), engine(spec, C, 4096)
    t = 0
    for k, n in enumerate([2048, 1024, 4096, 1024]):
        if k == 2:
            a.reset_channels(np.arange(C))
            b.reset_state()
        x = S.noise(C, n, sample_offset=t)
        ya, yb = a.process([x])[0], b.process([x])[0]
        if spec_name == "config3":
            assert_bit_exact(ya, yb, f"call {k}")
        else:
            assert_bit_exact(ya[:, :299 if k == 2 else 0], yb[:, :299 if k == 2 else 0], f"call {k} warm-up")
            assert_audio_close(ya, yb, what=f"call {k}")
        t += n


def test_empty_list_first_call_reset_and_dropped_requests_are_no_ops():
    spec = S.target_chain(300)
    plain, empty, first, dropped, state = (engine(spec, C, 4096) for _ in range(5))
    empty.reset_channels([])
    first.reset_channels(R1)                 # before the first call: every channel is fresh anyway
    t = 0
    for k, n in enumerate([2048, 1024, 4096]):
        if k == 1:
            dropped.reset_channels(R1)       # a pending reset followed by reset_state is reset_state alone
            dropped.reset_state()
            state.reset_state()
        x = S.noise(C, n, sample_offset=t)
        y = plain.process([x])[0]
        launches = plain.kernel_launches
        assert_bit_exact(empty.process([x])[0], y, f"empty list, call {k}")
        assert empty.kernel_launches == launches
        assert_bit_exact(first.process([x])[0], y, f"reset before the first call, call {k}")
        yd, ys = dropped.process([x])[0], state.process([x])[0]
        assert_bit_exact(yd, ys, f"pending reset then reset_state, call {k}")
        assert dropped.kernel_launches == state.kernel_launches
        t += n


def _device_run(e, xs, resets, stream):
    import torch

    outs = []
    with torch.cuda.stream(stream):
        for k, x in enumerate(xs):
            if k in resets:
                e.reset_channels(resets[k])
            xi = torch.from_numpy(x).cuda()
            yo = torch.empty_like(xi)
            e.process_device([xi], [yo], x.shape[1], stream=stream)
            outs.append(yo)
    stream.synchronize()
    return [y.cpu().numpy() for y in outs]


@pytest.mark.parametrize("channels,chunks", [(C, None), (160, "2")])
def test_device_pointers_on_a_side_stream_and_device_chunks(monkeypatch, channels, chunks):
    """The clear is enqueued on the caller's stream in front of the fork of the device chunks: the same outputs as the host
    path."""
    import torch

    spec = S.target_chain(300)
    calls = [2048, 1024, 4096, 1024]
    resets = {1: R1, 2: [0, 33, 100, 159] if channels == 160 else R2, 3: R3}
    xs = [S.noise(channels, n, seed=4, sample_offset=sum(calls[:k])) for k, n in enumerate(calls)]
    if chunks:
        monkeypatch.setenv("DSPB_CHUNKS", chunks)
    dev = engine(spec, channels, 4096)
    if chunks:
        monkeypatch.delenv("DSPB_CHUNKS")
    host = engine(spec, channels, 4096)
    got = _device_run(dev, xs, resets, torch.cuda.Stream())
    for k, x in enumerate(xs):
        if k in resets:
            host.reset_channels(resets[k])
        assert_bit_exact(got[k], host.process([x])[0], f"device vs host call {k}")


def test_async_host_path_reset_between_in_flight_calls():
    import torch

    spec = S.target_chain(300)
    calls = [2048, 2048, 2048, 2048]
    resets = {1: R1, 2: R2, 3: R3}
    xs = [S.noise(C, n, seed=6, sample_offset=sum(calls[:k])) for k, n in enumerate(calls)]
    blocking, asy = engine(spec, C, 2048), engine(spec, C, 2048)
    want = []
    for k, x in enumerate(xs):
        if k in resets:
            blocking.reset_channels(resets[k])
        want.append(blocking.process([x])[0])
    pinned = []
    for k, x in enumerate(xs):
        if k in resets:
            asy.reset_channels(resets[k])    # the previous call is still in flight
        xi, yo = torch.from_numpy(x).pin_memory(), torch.empty((C, x.shape[1]), dtype=torch.float32).pin_memory()
        asy.process_host([xi], [yo], x.shape[1], wait=False)
        pinned.append((xi, yo))
    asy.sync()
    for k, (_, yo) in enumerate(pinned):
        assert_bit_exact(yo.numpy(), want[k], f"async call {k}")


def test_scan_mode_filter(oracle_mod):
    spec = chain("biquad", **S.rbj_biquad("lp", 1000.0))
    e = engine(spec, C, max(CALLS), iir_mode=1)
    assert "time-parallel scan (probe error" in e.describe_plan()
    ref = Ref(oracle_mod, spec, C)
    t = 0
    for k, n in enumerate(CALLS):
        if k in RESETS:
            e.reset_channels(RESETS[k])
            ref.start(RESETS[k])
        x = S.noise(C, n, sample_offset=t)
        got, want = e.process([x])[0], ref.process(x, n)
        for g in ref.groups():
            assert_audio_close(got[g], want[g], what=f"scan call {k} channels {g[:4]}...")
        t += n


def _launches(e, x, n):
    import torch

    xi = torch.from_numpy(x).cuda()
    yo = torch.empty_like(xi)
    e.process_device([xi], [yo], n)
    torch.cuda.synchronize()
    return e.kernel_launches


@pytest.mark.parametrize("N,n,patched_calls", [(300, 2048, 1), (4096, 1024, 4)])
def test_launch_counts(N, n, patched_calls):
    """Nothing pending and no channel in its own warm-up: exactly the twin's launches.  The call after a reset: one clear
    launch more, and one patch launch per FIR step (one launch range here) while a reset channel is in its warm-up."""
    spec = S.target_chain(N)
    e, twin = engine(spec, C, n), engine(spec, C, n)
    calls = 4 + 4096 // n + patched_calls + 1
    for k in range(calls):
        x = S.noise(C, n, sample_offset=k * n)
        if k == 4 + 4096 // n:
            e.reset_channels(R1)
        le, lt = _launches(e, x, n), _launches(twin, x, n)
        j = k - (4 + 4096 // n)
        extra = (1 if j == 0 else 0) + (1 if 0 <= j < patched_calls else 0)
        assert le == lt + extra, f"call {k}: {le} launches, twin {lt}, expected +{extra}"
