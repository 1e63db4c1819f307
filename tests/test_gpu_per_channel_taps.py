"""Per-channel FIR impulse responses (dspb_node_set_taps_channels) on the GPU.

Reference: the channels are grouped by their impulse response and one Oracle per group runs exactly the channels that use it,
with plain set_taps.  The FFT path must be within the parity tolerance (each group against its own level); the warm-up
samples (the first N - 1 since reset, recomputed by the direct kernel) and everything of fir_mode = 1 and of impulse
responses past the FFT kernels (5000 taps) must be bit-exact.
"""
import numpy as np
import pytest

from dsp_stuff_b200 import GraphSpec
from dsp_stuff_b200 import signals as S
from tests.util import assert_audio_close, assert_bit_exact, make_oracle

pytestmark = pytest.mark.gpu
FIR_FFT, FIR_DIRECT = 0, 1
FIR = 0   # the fir node of S.config4
# wide + narrow segments (24576, 16384, ragged 128 * 88, 128 * 8) and UPC calls (1024, 2048) in between, so the UPC
# delay line is re-primed after every segment call
CALLS = [1024, 2048, 24576, 1024, 128 * 88, 16384, 2048, 128 * 8]


def irs(K, N, seed=0):
    """K decaying random impulse responses (rows of taps, i.e. reversed like set_taps), peak about 0.1."""
    rng = np.random.default_rng(seed)
    env = np.exp(-np.arange(N) / (N / 4.0 + 1.0))
    return (rng.standard_normal((K, N)) * env * 0.1)[:, ::-1].copy()


def assign(kind, C, K):
    c = np.arange(C)
    return {"interleaved": c % K, "contiguous": c * K // C, "distinct": c}[kind].astype(np.int32)


class GroupedTaps:
    """One Oracle per distinct (set, extra parameters) key; each runs exactly its channels with plain set_taps."""

    def __init__(self, oracle_mod, spec, bank, idx, node=FIR, f32=None):
        f32 = f32 or {}
        keys = [(int(idx[c]),) + tuple(float(v[c]) for v in f32.values()) for c in range(len(idx))]
        self.C = len(idx)
        self.parts = []
        for key in dict.fromkeys(keys):
            sel = np.array([c for c in range(self.C) if keys[c] == key])
            o = make_oracle(oracle_mod, spec, len(sel))
            o.set_taps(node, bank[key[0]])
            for (nid, field), val in zip(f32, key[1:]):
                o.set_f32(nid, field, val)
            self.parts.append((sel, o))

    def process(self, x):
        out = np.zeros_like(x)
        for sel, o in self.parts:
            out[sel] = o.process([x[sel]])[0]
        return out

    def reset_state(self):
        for _, o in self.parts:
            o.reset_state()


def engine(spec, C, n, fir_mode=FIR_FFT, **kw):
    from dsp_stuff_b200.engine import Engine

    e = Engine(C, block=128, max_samples=n, fir_mode=fir_mode, **kw)
    spec.apply(e)
    return e


def check(got, ref, parts, N, started, exact, what):
    """got / ref: [C x n] of one call that starts `started` samples after reset."""
    if exact:
        assert_bit_exact(got, ref, what)
        return
    warm = max(0, min(got.shape[1], N - 1 - started))
    if warm:
        assert_bit_exact(got[:, :warm], ref[:, :warm], f"{what} warm-up")
    for sel, _ in parts:
        assert_audio_close(got[sel], ref[sel], what=f"{what} channels {sel[:3]}...")


def run_calls(e, ref, C, N, calls, exact, what, seed=0):
    started = 0
    for k, n in enumerate(calls):
        x = S.noise(C, n, seed=seed, sample_offset=started)
        got = e.process([x])[0]
        check(got, ref.process(x), ref.parts, N, started, exact, f"{what} call {k} (n={n})")
        started += n


CASES = [  # (n_taps, channels, assignment, fir_mode)
    (1, 5, "distinct", FIR_FFT),
    (300, 33, "interleaved", FIR_FFT),
    (300, 64, "contiguous", FIR_FFT),
    (300, 64, "distinct", FIR_FFT),
    (4096, 33, "interleaved", FIR_FFT),
    (4096, 64, "distinct", FIR_FFT),
    (4097, 33, "contiguous", FIR_FFT),      # the longest impulse response of the FFT kernels (no UPC)
    (5000, 5, "interleaved", FIR_FFT),      # past the FFT kernels: the exact direct path, bit for bit
    (300, 33, "interleaved", FIR_DIRECT),
    (4096, 5, "distinct", FIR_DIRECT),
]


@pytest.mark.parametrize("N,C,kind,fir_mode", CASES, ids=[f"N{n}-C{c}-{k}-mode{m}" for n, c, k, m in CASES])
def test_against_grouped_oracle(oracle_mod, N, C, kind, fir_mode):
    K = min(C, 3 if kind != "distinct" else C)
    bank, idx = irs(K, N, seed=N), assign(kind, C, K)
    spec = S.config4(N)
    e = engine(spec, C, max(CALLS), fir_mode=fir_mode)
    e.set_taps_channels(FIR, bank, idx)
    ref = GroupedTaps(oracle_mod, spec, bank, idx)
    exact = fir_mode == FIR_DIRECT or N > 4097
    run_calls(e, ref, C, N, CALLS, exact, f"N={N} C={C} {kind}")


def test_average_mode_and_impulse_response_form(oracle_mod):
    C, N = 33, 300
    bank, idx = irs(4, N, seed=7), assign("interleaved", C, 4)
    spec = GraphSpec().node(10, "input").node(0, "fir", mode="Average", taps=[1.0]).node(11, "output")
    spec.link(10, "out", 0, "in").link(0, "out", 11, "in")
    e = engine(spec, C, 24576)
    e.set_impulse_response_channels(0, bank[:, ::-1], idx)     # rows in time order: reversed per row
    ref = GroupedTaps(oracle_mod, spec, bank, idx, node=0)
    run_calls(e, ref, C, N, [1024, 24576, 2048], False, "Average")


def test_reset_state(oracle_mod):
    C, N = 33, 300
    bank, idx = irs(C, N, seed=2), assign("distinct", C, C)
    spec = S.config4(N)
    e = engine(spec, C, 24576)
    e.set_taps_channels(FIR, bank, idx)
    ref = GroupedTaps(oracle_mod, spec, bank, idx)
    run_calls(e, ref, C, N, [2048, 128 * 88], False, "before reset")
    e.reset_state()
    ref.reset_state()
    run_calls(e, ref, C, N, [1024, 16384, 1024], False, "after reset", seed=5)


def test_target_chain_with_per_channel_gain(oracle_mod):
    C, N = 64, 256
    g = S.target_chain(N)
    bank, idx = irs(4, N, seed=3), assign("interleaved", C, 4)
    level = np.array([0.5, 1.0, 2.0])[np.arange(C) % 3].astype(np.float32)
    e = engine(g, C, 4096)
    e.set_taps_channels(4, bank, idx)
    e.set_f32_channels(0, "level", level)
    ref = GroupedTaps(oracle_mod, g, bank, idx, node=4, f32={(0, "level"): level})
    run_calls(e, ref, C, N, [2048, 4096, 1024], False, "target chain")


def _device_process(e, x):
    import torch

    xi = torch.from_numpy(x).cuda()
    yo = torch.empty_like(xi)
    e.process_device([xi], [yo], x.shape[1])
    torch.cuda.synchronize()
    return yo.cpu().numpy()


def test_device_chunks_host_and_async_paths_agree(oracle_mod, monkeypatch):
    """Device-pointer chunks (DSPB_CHUNKS=4, set before the engine is created), the host path and the asynchronous host
    path run the same transform-table slices: bit-identical outputs, and within tolerance of the oracle."""
    import torch

    C, N = 256, 300
    g = S.target_chain(N)
    bank, idx = irs(C, N, seed=4), assign("distinct", C, C)
    calls = [1024, 4096, 2048, 4096]
    xs = [S.noise(C, n, seed=9, sample_offset=sum(calls[:k])) for k, n in enumerate(calls)]
    monkeypatch.setenv("DSPB_CHUNKS", "4")
    chunked = engine(g, C, 4096)
    chunked.set_taps_channels(4, bank, idx)
    monkeypatch.delenv("DSPB_CHUNKS")
    host, asy = engine(g, C, 4096), engine(g, C, 4096)
    host.set_taps_channels(4, bank, idx)
    asy.set_taps_channels(4, bank, idx)
    ref = GroupedTaps(oracle_mod, g, bank, idx, node=4)
    pinned = []
    for k, x in enumerate(xs):
        a = _device_process(chunked, x)
        b = host.process([x])[0]
        assert_bit_exact(a, b, f"chunked device vs host call {k}")
        check(b, ref.process(x), ref.parts, N, sum(calls[:k]), False, f"host call {k}")
        xi, yo = torch.from_numpy(x).pin_memory(), torch.empty((C, x.shape[1]), dtype=torch.float32).pin_memory()
        asy.process_host([xi], [yo], x.shape[1], wait=False)
        pinned.append((xi, yo, b))
    asy.sync()
    for k, (_, yo, b) in enumerate(pinned):
        assert_bit_exact(yo.numpy(), b, f"async host call {k}")


def test_node_process(oracle_mod):
    C, N, n = 33, 300, 2048
    bank, idx = irs(3, N, seed=6), assign("interleaved", C, 3)
    g = GraphSpec().node(0, "fir", mode="Balanced", taps=[1.0])
    e = engine(g, C, n)
    e.set_taps_channels(0, bank, idx)
    ref = GroupedTaps(oracle_mod, g, bank, idx, node=0)
    for call in range(2):
        x = S.noise(C, n, sample_offset=call * n)
        got = e.node_process(0, [x])[0]
        want = np.zeros_like(got)
        for sel, o in ref.parts:
            want[sel] = o.node_process(0, [x[sel]])[0]
        check(got, want, ref.parts, N, call * n, False, f"node_process call {call}")


def test_even_contiguous_runs_match_shared_engines_bit_for_bit():
    """Sets in contiguous runs of even length that start on even channels pair exactly like shared taps: every row is
    bit-identical to a shared engine holding that row's taps."""
    C, N = 64, 300
    runs = [0] * 6 + [1] * 10 + [2] * 16 + [3] * 2 + [0] * 30       # set 0 twice; every run even, on even channels
    idx = np.array(runs, dtype=np.int32)
    bank = irs(4, N, seed=8)
    spec = S.config4(N)
    e = engine(spec, C, 24576)
    e.set_taps_channels(FIR, bank, idx)
    shared = []
    for k in range(4):
        s = engine(spec, C, 24576)
        s.set_taps(FIR, bank[k])
        shared.append(s)
    started = 0
    for n in [1024, 24576, 2048, 128 * 88]:
        x = S.noise(C, n, sample_offset=started)
        got = e.process([x])[0]
        for k, s in enumerate(shared):
            sel = np.flatnonzero(idx == k)
            assert_bit_exact(got[sel], s.process([x])[0][sel], f"set {k} n={n}")
        started += n


@pytest.mark.parametrize("world", [1, 2, 4])
def test_shards_on_32_channel_boundaries_equal_the_whole_run(world):
    from dsp_stuff_b200.shard import channel_range

    C, N = 128, 300
    bank, idx = irs(7, N, seed=10), (np.arange(C) * 5 % 7).astype(np.int32)
    spec = S.config4(N)
    whole = engine(spec, C, 24576)
    whole.set_taps_channels(FIR, bank, idx)
    shards = []
    for r in range(world):
        lo, hi = channel_range(r, world, C)
        assert lo % 32 == 0
        s = engine(spec, hi - lo, 24576)
        s.set_taps_channels(FIR, bank, idx[lo:hi])
        shards.append((lo, hi, s))
    started = 0
    for n in [2048, 24576, 1024]:
        x = S.noise(C, n, sample_offset=started)
        ref = whole.process([x])[0]
        for lo, hi, s in shards:
            assert_bit_exact(s.process([np.ascontiguousarray(x[lo:hi])])[0], ref[lo:hi], f"shard [{lo}, {hi}) n={n}")
        started += n


@pytest.mark.parametrize("kind", ["distinct", "bank8"])
def test_fft_matches_direct_at_full_width(kind):
    """4096 x 24576: the FFT path with 4096 distinct impulse responses or an 8-set bank against the bit-exact direct path
    on every 257th channel."""
    C, N, n = 4096, 4096, 24576
    K = C if kind == "distinct" else 8
    bank, idx = irs(K, N, seed=11), assign("distinct" if kind == "distinct" else "interleaved", C, K)
    spec = S.config4(N)
    x = S.noise(C, n)
    e = engine(spec, C, n)
    e.set_taps_channels(FIR, bank, idx)
    a = e.process([x])[0]
    sel = np.arange(0, C, 257)
    d = engine(spec, len(sel), n, fir_mode=FIR_DIRECT)
    d.set_taps_channels(FIR, bank, idx[sel])
    b = d.process([np.ascontiguousarray(x[sel])])[0]
    assert_bit_exact(a[sel, :N - 1], b[:, :N - 1], "warm-up")
    for i in range(len(sel)):
        assert_audio_close(a[sel[i]], b[i], what=f"channel {sel[i]}")
