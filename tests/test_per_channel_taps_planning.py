"""Per-channel FIR impulse responses (dspb_node_set_taps_channels) in planning mode (device -1, no GPU): argument checks,
the collapse of identical rows to the shared case, deduplication, the transform counts of the pairing rule in the plan
listing, and set_taps returning the node to shared taps.  The numeric side is tests/test_gpu_per_channel_taps.py."""
import re

import numpy as np
import pytest

from dsp_stuff_b200 import GraphSpec
from dsp_stuff_b200 import signals as S
from dsp_stuff_b200.engine import FIR_DIRECT, FIR_FFT, FIR_FFT_PACKED, FIR_TOEPLITZ, Engine, EngineError

ERR_INVALID, ERR_UNKNOWN_NODE = -1, -2
FIR = 4   # the fir node of S.target_chain


def planning_engine(channels, n_taps=64, fir_mode=FIR_FFT):
    e = Engine(channels, block=128, max_samples=128 * 9, device=-1, fir_mode=fir_mode)
    S.target_chain(n_taps).apply(e)
    return e


def bank(k, n, seed=0):
    return np.random.default_rng(seed).standard_normal((k, n)) * 0.05


def fir_line(e):
    return next(line for line in e.describe_plan().splitlines() if "fir step" in line)


def counts(e):
    m = re.search(r"per-channel taps: (\d+) sets(?:, (\d+) transforms \((\d+) single-channel\))?", fir_line(e))
    return None if m is None else tuple(int(g) if g is not None else None for g in m.groups())


def test_error_codes():
    C, N = 8, 64
    e = planning_engine(C, N)
    b, idx = bank(2, N), np.arange(C, dtype=np.int32) % 2
    with pytest.raises(EngineError) as ei:
        e.set_taps_channels(77, b, idx)
    assert ei.value.code == ERR_UNKNOWN_NODE
    with pytest.raises(EngineError) as ei:
        e.set_taps_channels(0, b, idx)                      # a gain node
    assert ei.value.code == ERR_INVALID and "not a fir" in str(ei.value)
    for bad in (idx[:-1], np.concatenate([idx, idx[:1]])):  # n_channels != channels
        with pytest.raises(EngineError) as ei:
            e.set_taps_channels(FIR, b, bad)
        assert ei.value.code == ERR_INVALID
    for v in (-1, 2):                                       # outside [0, n_sets)
        bad = idx.copy()
        bad[5] = v
        with pytest.raises(EngineError) as ei:
            e.set_taps_channels(FIR, b, bad)
        assert ei.value.code == ERR_INVALID and "set_index[5]" in str(ei.value)
    L = e._L
    for fn in (L.dspb_node_set_taps_channels, L.dspb_node_set_impulse_response_channels):
        assert fn(e._h, FIR, None, 2, N, idx.ctypes.data, C) == ERR_INVALID
        assert fn(e._h, FIR, b.ctypes.data, 2, N, None, C) == ERR_INVALID
        assert fn(e._h, FIR, b.ctypes.data, 0, N, idx.ctypes.data, C) == ERR_INVALID
        assert fn(e._h, FIR, b.ctypes.data, 2, 0, idx.ctypes.data, C) == ERR_INVALID
        assert fn(None, FIR, b.ctypes.data, 2, N, idx.ctypes.data, C) == ERR_INVALID
    # the failed calls changed nothing
    assert counts(e) is None


@pytest.mark.parametrize("mode", [FIR_TOEPLITZ, FIR_FFT_PACKED])
def test_distinct_sets_need_fft_or_direct_mode(mode):
    C, N = 8, 64
    e = planning_engine(C, N, fir_mode=mode)
    shared = e.describe_plan()
    with pytest.raises(EngineError) as ei:
        e.set_taps_channels(FIR, bank(2, N), np.arange(C) % 2)
    assert ei.value.code == ERR_INVALID and "fir_mode 0 or 1" in str(ei.value)
    # identical rows are the shared case in every mode
    b = bank(1, N)
    e.set_taps_channels(FIR, np.concatenate([b, b]), np.arange(C) % 2)
    e.compile()
    ref = planning_engine(C, N, fir_mode=mode)
    ref.set_taps(FIR, b[0])
    ref.compile()
    assert e.describe_plan() == ref.describe_plan() == shared   # the listing names the tap count, not the values


@pytest.mark.parametrize("mode", [FIR_FFT, FIR_DIRECT, FIR_TOEPLITZ, FIR_FFT_PACKED])
def test_all_equal_rows_are_the_shared_case_byte_for_byte(mode):
    C, N = 64, 300
    b = bank(1, N, seed=3)
    ref = planning_engine(C, N, fir_mode=mode)
    ref.set_taps(FIR, b[0])
    ref.compile()
    e = planning_engine(C, N, fir_mode=mode)
    e.set_taps_channels(FIR, np.repeat(b, 5, axis=0), np.arange(C) % 5)   # five copies of one row
    e.compile()
    assert e.describe_plan() == ref.describe_plan()
    assert e.get_i64(FIR, "n_taps") == N
    # the impulse-response form reverses each row
    e.set_impulse_response_channels(FIR, np.repeat(b[:, ::-1], 3, axis=0), np.arange(C) % 3)
    e.compile()
    assert e.describe_plan() == ref.describe_plan()
    if mode in (FIR_FFT, FIR_DIRECT):   # -0.0 and +0.0 differ in their bits: two sets
        z = np.repeat(b, 2, axis=0)
        z[0, 7], z[1, 7] = 0.0, -0.0
        e.set_taps_channels(FIR, z, np.arange(C) % 2)
        e.compile()
        assert counts(e)[0] == 2


def test_identical_and_unused_rows_are_dropped():
    C, N = 64, 128
    b = bank(6, N, seed=1)
    b[4] = b[1]                                       # row 4 repeats row 1
    idx = np.array([0, 1, 4, 2] * (C // 4), dtype=np.int32)   # rows 3 and 5 unused
    e = planning_engine(C, N)
    e.set_taps_channels(FIR, b, idx)
    e.compile()
    k, xf, single = counts(e)
    assert k == 3
    # per 32-group: set 0 (rows 0) 8 channels, set 1 (rows 1 and 4) 16, set 2 (row 2) 8: all even
    assert (xf, single) == (32, 0)


def model_transforms(idx):
    """The pairing rule restated: per aligned 32-channel group, per set, ceil(channels / 2) transforms, odd ones single."""
    total = single = 0
    for g0 in range(0, len(idx), 32):
        for k in np.unique(idx[g0:g0 + 32]):
            m = int(np.sum(idx[g0:g0 + 32] == k))
            total += (m + 1) // 2
            single += m % 2
    return total, single


@pytest.mark.parametrize("C,assign,expect", [
    (64, "mod8", (8, 32, 0)),         # 4 channels of each set per 32-group: the shared case's 32 transforms
    (64, "distinct", (64, 64, 64)),   # one channel per transform
    (64, "runs8", (8, 32, 0)),        # contiguous runs of 8
    (64, "runs3", (22, 43, 22)),      # runs of 3: every run leaves one channel alone (the run over channel 32 two)
    (33, "mod8", (8, 17, 1)),         # group 0: 4 per set -> 16; group 1: channel 32 alone
    (33, "mod2", (2, 17, 1)),         # group 0: 16 per set -> 16; group 1: channel 32 alone
    (33, "distinct", (33, 33, 33)),
    (5, "mod2", (2, 3, 1)),           # set 0 has channels 0, 2, 4 -> 2 transforms, set 1: 1, 3 -> 1
    (4096, "mod8", (8, 2048, 0)),     # full width: as many transforms as shared taps
    (4096, "distinct", (4096, 4096, 4096)),
])
def test_transform_counts(C, assign, expect):
    c = np.arange(C)
    idx = {"mod8": c % 8, "mod2": c % 2, "distinct": c, "runs8": c // 8, "runs3": c // 3}[assign]
    e = planning_engine(C, 256)
    e.set_taps_channels(FIR, bank(int(idx.max()) + 1, 256), idx)
    e.compile()
    assert counts(e) == expect, fir_line(e)
    assert expect[1:] == model_transforms(idx)


@pytest.mark.parametrize("seed", range(6))
def test_random_assignments_match_the_pairing_model(seed):
    rng = np.random.default_rng(seed)
    C = int(rng.integers(2, 300))
    K = int(rng.integers(2, 12))
    idx = rng.integers(0, K, C).astype(np.int32)
    if len(np.unique(idx)) < 2:
        idx[0] = (idx[0] + 1) % K
    e = planning_engine(C, 64)
    e.set_taps_channels(FIR, bank(K, 64, seed), idx)
    e.compile()
    assert counts(e) == (len(np.unique(idx)),) + model_transforms(idx)


def test_direct_path_lists_sets_only():
    C = 16
    for mode, n in ((FIR_DIRECT, 64), (FIR_FFT, 5000)):       # 5000 taps: past the FFT kernels, the exact path runs
        e = planning_engine(C, n, fir_mode=mode)
        e.set_taps_channels(FIR, bank(4, n), np.arange(C) % 4)
        e.compile()
        assert counts(e) == (4, None, None), fir_line(e)


def test_set_taps_returns_to_the_shared_listing():
    C, N = 64, 64
    e = planning_engine(C, N)
    e.set_taps(FIR, bank(1, N)[0])
    e.compile()
    shared = e.describe_plan()
    e.set_taps_channels(FIR, bank(8, N), np.arange(C) % 8)
    e.compile()
    assert e.describe_plan() != shared and counts(e) == (8, 32, 0)
    e.set_taps(FIR, bank(1, N)[0])
    e.compile()
    assert e.describe_plan() == shared
    e.set_impulse_response_channels(FIR, bank(8, N), np.arange(C) % 8)
    e.compile()
    assert counts(e) == (8, 32, 0)
    e.set_impulse_response(FIR, bank(1, N)[0][::-1])
    e.compile()
    assert e.describe_plan() == shared


def test_epilogue_and_per_channel_gain_listed_together():
    """The FIR step keeps its fused sink epilogue; per-channel f32 values and per-channel taps coexist."""
    C, N = 64, 64
    g = GraphSpec().node(10, "input").node(0, "gain").node(1, "fir", taps=[1.0]).node(11, "output")
    g.link(10, "out", 0, "in").link(0, "out", 1, "in").link(1, "out", 11, "in")
    e = Engine(C, block=128, max_samples=128 * 9, device=-1)
    g.apply(e)
    e.set_f32_channels(0, "level", np.linspace(0.5, 1.5, C))
    e.set_taps_channels(1, bank(2, N), np.arange(C) % 2)
    e.compile()
    line = next(x for x in e.describe_plan().splitlines() if "fir step" in x)
    assert "per-channel taps: 2 sets, 32 transforms (0 single-channel), epilogue" in line
    assert "per-channel[level]" in e.describe_plan()
