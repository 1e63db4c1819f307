"""Per-channel state reset (dspb_reset_channels) in planning mode (device -1, no GPU): the error codes and the order of the
checks, nothing recorded by a failed call, deduplication of the recorded channels, the NULL list with zero channels, and the
exported symbol.  The numeric side is tests/test_gpu_reset_channels.py."""
import ctypes

import numpy as np
import pytest

from dsp_stuff_b200 import signals as S
from dsp_stuff_b200.engine import Engine, EngineError

ERR_INVALID = -1
C = 70


def planning_engine():
    e = Engine(C, block=128, max_samples=1024, device=-1)
    S.target_chain(64).apply(e)
    return e


def pending(e):
    return e.get_i64(0, "pending_resets")


def call(h, channels, n):
    from dsp_stuff_b200.engine import load_library

    return load_library().dspb_reset_channels(h, channels, n)


def test_symbol_is_exported():
    e = planning_engine()
    assert hasattr(e._L, "dspb_reset_channels")


def test_error_codes_and_their_order():
    e = planning_engine()
    ok = np.array([0, 5], dtype=np.int32)
    bad = np.array([0, C], dtype=np.int32)
    assert call(None, ok.ctypes.data, 2) == ERR_INVALID                 # null engine first, whatever else is wrong
    assert call(None, None, -1) == ERR_INVALID
    assert call(e._h, None, -1) == ERR_INVALID                           # n < 0 before the null list
    assert "n_channels" in e._L.dspb_last_error().decode()
    assert call(e._h, None, 3) == ERR_INVALID                            # null list with n > 0
    assert "null" in e._L.dspb_last_error().decode()
    assert call(e._h, bad.ctypes.data, 2) == ERR_INVALID                 # index == channels
    assert "channels[1]" in e._L.dspb_last_error().decode()
    for v in (-1, C, 1 << 30):
        with pytest.raises(EngineError) as ei:
            e.reset_channels([3, v])
        assert ei.value.code == ERR_INVALID and "channels[1]" in str(ei.value)
    assert pending(e) == 0                                               # no failed call recorded anything


def test_failed_call_records_nothing_even_with_valid_leading_indices():
    e = planning_engine()
    e.reset_channels([1, 2])
    with pytest.raises(EngineError):
        e.reset_channels([3, 4, C])          # 3 and 4 are valid, the call fails as a whole
    assert pending(e) == 2
    e.reset_channels([4])                    # a later valid call sees only what the good calls recorded
    assert pending(e) == 3


def test_zero_channels_is_a_no_op_and_null_is_accepted():
    e = planning_engine()
    assert call(e._h, None, 0) == 0
    e.reset_channels(np.zeros(0, dtype=np.int32))
    assert pending(e) == 0


def test_requests_accumulate_deduplicated():
    e = planning_engine()
    e.reset_channels([0, 69, 31, 32, 31, 0])
    assert pending(e) == 4
    e.reset_channels(np.array([32, 33, 69], dtype=np.int32))
    assert pending(e) == 5
    e.reset_channels(np.arange(C, dtype=np.int32))
    assert pending(e) == C


def test_python_binding_takes_any_integer_sequence():
    e = planning_engine()
    e.reset_channels(np.array([7, 8], dtype=np.int64))
    e.reset_channels((9,))
    assert pending(e) == 3
    assert e._L.dspb_reset_channels.argtypes == [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64]
