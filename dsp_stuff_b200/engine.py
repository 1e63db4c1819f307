"""Host-side mirror of the reference's node/graph interface, over the C ABI (include/dspb200.h).

The reference drives nodes through `Node`/`NodeStatic`/`SimpleNode` (dsp-stuff/src/node.rs:104-146)
and wires them in `UiContext` (runtime.rs:125-224).  `Engine` keeps those names and meanings:
typenames are the `cfg_name` strings (nodes/mod.rs:92-123), fields and ports are the Rust
identifiers, enum values are variant names, errors surface where the reference would panic.

PyTorch is used only for device memory and streams.  There is NO CPU fallback: the constructor
raises if libdspb200.so is missing or no CUDA device is usable.
"""
from __future__ import annotations

import ctypes
import os
from typing import List, Optional, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libdspb200.so")

MEM_DEVICE = 0
MEM_HOST = 1
MEM_HOST_ASYNC = 2
FIR_FFT = 0
FIR_DIRECT = 1
FIR_TOEPLITZ = 2
FIR_FFT_PACKED = 3


class Config(ctypes.Structure):
    _fields_ = [
        ("channels", ctypes.c_int32),
        ("block", ctypes.c_int32),
        ("sample_rate", ctypes.c_int32),
        ("ref_block", ctypes.c_int32),
        ("ring_granule", ctypes.c_int32),
        ("device", ctypes.c_int32),
        ("max_samples", ctypes.c_int64),
        ("fir_fft_log2", ctypes.c_int32),
        ("fir_mode", ctypes.c_int32),
        ("iir_mode", ctypes.c_int32),
    ]


class EngineError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"dspb200 error {code}: {msg}")
        self.code = code


# Every symbol include/dspb200.h declares (checked by tests/test_abi.py against the header text).
ABI_SYMBOLS = [
    "dspb_engine_create", "dspb_engine_destroy", "dspb_last_error", "dspb_abi_version", "dspb_node_add",
    "dspb_node_set_f32", "dspb_node_set_enum", "dspb_node_set_taps", "dspb_node_set_impulse_response", "dspb_link",
    "dspb_load_graph_json", "dspb_compile", "dspb_process", "dspb_node_process", "dspb_reset_state",
    "dspb_node_get_i64", "dspb_node_port_index", "dspb_describe_plan", "dspb_profile_enable", "dspb_profile_read",
    "dspb_fold_stereo", "dspb_dup_stereo", "dspb_resample_dup_stereo", "dspb_sync", "dspb_node_set_f32_channels",
    "dspb_node_set_taps_channels", "dspb_node_set_impulse_response_channels",
]

_lib = None


def load_library(path: Optional[str] = None):
    """Loads libdspb200.so; raises (never falls back) when it has not been built."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or _LIB_PATH
    if not os.path.exists(p):
        raise EngineError(-5, f"{p} not found: build it with `python -m dsp_stuff_b200.build` (no CPU fallback exists)")
    L = ctypes.CDLL(p)
    vp, i64, cp = ctypes.c_void_p, ctypes.c_int64, ctypes.c_char_p
    L.dspb_last_error.restype = cp
    L.dspb_engine_create.argtypes = [ctypes.POINTER(Config), ctypes.POINTER(vp)]
    L.dspb_engine_destroy.argtypes = [vp]
    L.dspb_engine_destroy.restype = None
    L.dspb_node_add.argtypes = [vp, cp, i64]
    L.dspb_node_set_f32.argtypes = [vp, i64, cp, ctypes.c_float]
    L.dspb_node_set_f32_channels.argtypes = [vp, i64, cp, vp, i64]
    L.dspb_node_set_enum.argtypes = [vp, i64, cp, cp]
    L.dspb_node_set_taps.argtypes = [vp, i64, vp, i64]
    L.dspb_node_set_impulse_response.argtypes = [vp, i64, vp, i64]
    L.dspb_node_set_taps_channels.argtypes = [vp, i64, vp, i64, i64, vp, i64]
    L.dspb_node_set_impulse_response_channels.argtypes = [vp, i64, vp, i64, i64, vp, i64]
    L.dspb_link.argtypes = [vp, i64, cp, i64, cp]
    L.dspb_load_graph_json.argtypes = [vp, cp]
    L.dspb_compile.argtypes = [vp]
    L.dspb_process.argtypes = [vp, vp, vp, i64, ctypes.c_int, vp]
    L.dspb_node_process.argtypes = [vp, i64, vp, vp, vp, i64, ctypes.c_int, vp]
    L.dspb_reset_state.argtypes = [vp]
    L.dspb_node_get_i64.argtypes = [vp, i64, cp, ctypes.POINTER(i64)]
    L.dspb_node_port_index.argtypes = [vp, i64, cp, ctypes.c_int, ctypes.POINTER(ctypes.c_int32)]
    L.dspb_profile_enable.argtypes = [vp, ctypes.c_int]
    L.dspb_profile_read.argtypes = [vp, vp, vp, ctypes.c_int]
    L.dspb_describe_plan.argtypes = [vp, vp, i64]
    L.dspb_fold_stereo.argtypes = [vp, vp, vp, i64, ctypes.c_int, vp]
    L.dspb_dup_stereo.argtypes = [vp, vp, vp, i64, ctypes.c_int, vp]
    L.dspb_resample_dup_stereo.argtypes = [vp, vp, vp, i64, i64, ctypes.c_double, ctypes.c_int, vp, ctypes.POINTER(i64)]
    L.dspb_sync.argtypes = [vp]
    L.dspb_describe_plan.restype = i64
    if path is None:
        _lib = L
    return L


class Engine:
    """One engine = one graph instantiated over `channels` mono streams on one GPU."""

    def __init__(self, channels: int, block: int = 128, max_samples: int = 0, ring_granule: int = 1024,
                 device: int = 0, fir_mode: int = FIR_FFT, sample_rate: int = 48000, iir_mode: int = 0):
        self._L = load_library()
        self.channels = channels
        self.device = device
        cfg = Config(channels=channels, block=block, sample_rate=sample_rate, ref_block=128, ring_granule=ring_granule,
                     device=device, max_samples=max_samples, fir_fft_log2=0, fir_mode=fir_mode, iir_mode=iir_mode)
        h = ctypes.c_void_p()
        self._h = None
        self._ck(self._L.dspb_engine_create(ctypes.byref(cfg), ctypes.byref(h)))
        self._h = h
        self._n_in = 0
        self._n_out = 0

    def _ck(self, rc: int):
        if rc != 0:
            raise EngineError(rc, self._L.dspb_last_error().decode(errors="replace"))

    def close(self):
        if getattr(self, "_h", None):
            self._L.dspb_engine_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- graph construction (names follow the reference) ------------------------------------------------
    def add_node(self, typename: str, node_id: int):
        self._ck(self._L.dspb_node_add(self._h, typename.encode(), node_id))
        if typename == "input":
            self._n_in += 1
        elif typename == "output":
            self._n_out += 1

    def set_f32(self, node_id: int, field: str, value: float):
        self._ck(self._L.dspb_node_set_f32(self._h, node_id, field.encode(), float(value)))

    def set_f32_channels(self, node_id: int, field: str, values):
        """One slider value per channel (float32, length `channels`): channel c runs as if set_f32(values[c]) had been
        called on an engine holding only channel c.  All values bit-identical = set_f32(values[0]); a later set_f32 on
        the field makes it shared again.  reverb.seconds cannot vary per channel."""
        v = np.ascontiguousarray(values, dtype=np.float32).reshape(-1)
        self._ck(self._L.dspb_node_set_f32_channels(self._h, node_id, field.encode(), v.ctypes.data, v.size))

    def set_enum(self, node_id: int, field: str, variant: str):
        self._ck(self._L.dspb_node_set_enum(self._h, node_id, field.encode(), variant.encode()))

    def set_taps(self, node_id: int, taps):
        t = np.ascontiguousarray(taps, dtype=np.float64)
        self._ck(self._L.dspb_node_set_taps(self._h, node_id, t.ctypes.data, t.size))

    def set_impulse_response(self, node_id: int, h):
        t = np.ascontiguousarray(h, dtype=np.float64)
        self._ck(self._L.dspb_node_set_impulse_response(self._h, node_id, t.ctypes.data, t.size))

    def set_taps_channels(self, node_id: int, bank, set_index):
        """Per-channel impulse responses: bank [K, N] float64 (rows reversed like set_taps), set_index [channels] int32.
        Channel c runs as if set_taps(bank[set_index[c]]) had been called on an engine holding only channel c.  Identical
        rows are one set; all channels alike = set_taps(row).  A later set_taps / set_impulse_response makes it shared."""
        self._set_bank(self._L.dspb_node_set_taps_channels, node_id, bank, set_index)

    def set_impulse_response_channels(self, node_id: int, bank, set_index):
        """Same as set_taps_channels with impulse responses in time order (each row reversed like set_impulse_response)."""
        self._set_bank(self._L.dspb_node_set_impulse_response_channels, node_id, bank, set_index)

    def _set_bank(self, fn, node_id, bank, set_index):
        b = np.ascontiguousarray(bank, dtype=np.float64)
        if b.ndim == 1:
            b = b.reshape(1, -1)
        s = np.ascontiguousarray(set_index, dtype=np.int32).reshape(-1)
        self._ck(fn(self._h, node_id, b.ctypes.data, b.shape[0], b.shape[1], s.ctypes.data, s.size))

    def link(self, src: int, out_port: str, dst: int, in_port: str):
        self._ck(self._L.dspb_link(self._h, src, out_port.encode(), dst, in_port.encode()))

    def compile(self):
        self._ck(self._L.dspb_compile(self._h))

    def load_graph_json(self, text: str):
        self._ck(self._L.dspb_load_graph_json(self._h, text.encode()))
        import json

        doc = json.loads(text)
        self._n_in = sum(1 for n in doc["nodes"] if n["typename"] == "input")
        self._n_out = sum(1 for n in doc["nodes"] if n["typename"] == "output")

    def reset_state(self):
        self._ck(self._L.dspb_reset_state(self._h))

    def get_i64(self, node_id: int, key: str) -> int:
        v = ctypes.c_int64()
        self._ck(self._L.dspb_node_get_i64(self._h, node_id, key.encode(), ctypes.byref(v)))
        return v.value

    def port_index(self, node_id: int, port: str, is_output: bool = False) -> int:
        v = ctypes.c_int32()
        self._ck(self._L.dspb_node_port_index(self._h, node_id, port.encode(), int(is_output), ctypes.byref(v)))
        return v.value

    def describe_plan(self) -> str:
        n = self._L.dspb_describe_plan(self._h, None, 0)
        buf = ctypes.create_string_buffer(int(n))
        self._L.dspb_describe_plan(self._h, buf, n)
        return buf.value.decode()

    def profile(self, on: bool = True):
        self._ck(self._L.dspb_profile_enable(self._h, int(on)))

    def profile_read(self):
        """-> list of (total_ms, rounds) per schedule step, measured with CUDA events on the launch stream."""
        cap = 64
        ms = (ctypes.c_double * cap)()
        rounds = (ctypes.c_int64 * cap)()
        n = self._L.dspb_profile_read(self._h, ms, rounds, cap)
        if n < 0:
            self._ck(n)
        return [(ms[i], rounds[i]) for i in range(min(n, cap))]

    def plan_steps(self):
        """Parses describe_plan(): per step its kind and ALGORITHMIC bytes per channel-sample
        (4 B per global f32 read or write, 8 B per Reverb ring; SURVEY.md section 8d / DESIGN.md)."""
        import re

        steps = []
        for line in self.describe_plan().splitlines():
            if line.startswith("["):
                m = re.search(r"alg_bytes=(\d+)", line)
                steps.append({"kind": "fir" if "fir step" in line else "fused", "alg_bytes": int(m.group(1)) if m else 0,
                              "text": line.split("] ", 1)[1]})
        return steps

    @property
    def kernel_launches(self) -> int:
        return self.get_i64(0, "kernel_launches")

    # ---- the hot path -----------------------------------------------------------------------------------
    def process_device(self, inputs: Sequence, outputs: Sequence, n_samples: int, stream=None):
        """inputs/outputs: CUDA float32 torch tensors [C, n] (contiguous).  Enqueues on `stream`
        (default: torch's current stream) and returns without synchronising."""
        import torch

        assert len(inputs) == self._n_in and len(outputs) == self._n_out
        for t in list(inputs) + list(outputs):
            assert t.is_cuda and t.dtype == torch.float32 and t.is_contiguous() and tuple(t.shape) == (self.channels, n_samples)
        st = stream if stream is not None else torch.cuda.current_stream(self.device)
        ip = (ctypes.c_void_p * max(1, len(inputs)))(*[t.data_ptr() for t in inputs])
        op = (ctypes.c_void_p * max(1, len(outputs)))(*[t.data_ptr() for t in outputs])
        self._ck(self._L.dspb_process(self._h, ip, op, n_samples, MEM_DEVICE, ctypes.c_void_p(st.cuda_stream)))

    def sync(self):
        """Waits for every process_host(..., wait=False) call."""
        self._ck(self._L.dspb_sync(self._h))

    def process_host(self, inputs: Sequence, outputs: Sequence, n_samples: int, wait: bool = True):
        """inputs/outputs: host float32 buffers [C, n] (numpy arrays or CPU torch tensors, pinned for
        full speed).  Copies in, runs and copies out (pipelined over channel chunks); blocks until done unless
        wait=False (DSPB_MEM_HOST_ASYNC: keep the buffers alive and untouched until sync())."""
        assert len(inputs) == self._n_in and len(outputs) == self._n_out

        def ptr(a):
            if isinstance(a, np.ndarray):
                assert a.dtype == np.float32 and a.flags.c_contiguous and a.shape == (self.channels, n_samples)
                return a.ctypes.data
            assert (not a.is_cuda) and a.is_contiguous() and tuple(a.shape) == (self.channels, n_samples)
            return a.data_ptr()

        ip = (ctypes.c_void_p * max(1, len(inputs)))(*[ptr(t) for t in inputs])
        op = (ctypes.c_void_p * max(1, len(outputs)))(*[ptr(t) for t in outputs])
        self._ck(self._L.dspb_process(self._h, ip, op, n_samples, MEM_HOST if wait else MEM_HOST_ASYNC, None))

    # ---- device-boundary format steps (devices.rs:244-262, 443-500) ---------------------------------------
    def fold_stereo(self, interleaved: np.ndarray) -> np.ndarray:
        """[C, n_frames, 2] interleaved stereo -> [C, n_frames] mono, a + b (host buffers)."""
        x = np.ascontiguousarray(interleaved, dtype=np.float32)
        assert x.ndim == 3 and x.shape[0] == self.channels and x.shape[2] == 2
        out = np.empty(x.shape[:2], dtype=np.float32)
        self._ck(self._L.dspb_fold_stereo(self._h, x.ctypes.data, out.ctypes.data, x.shape[1], MEM_HOST, None))
        return out

    def dup_stereo(self, mono: np.ndarray) -> np.ndarray:
        """[C, n_frames] mono -> [C, n_frames, 2] interleaved stereo, both slots = the mono sample (host buffers)."""
        x = np.ascontiguousarray(mono, dtype=np.float32)
        assert x.ndim == 2 and x.shape[0] == self.channels
        out = np.empty(x.shape + (2,), dtype=np.float32)
        self._ck(self._L.dspb_dup_stereo(self._h, x.ctypes.data, out.ctypes.data, x.shape[1], MEM_HOST, None))
        return out

    def resample_dup_stereo(self, mono: np.ndarray, n_out: int, target_hz: float):
        """[C, n_in] mono at the engine rate -> ([C, n_out, 2] interleaved stereo at target_hz, consumed input samples):
        the playback callback's sinc converter + duplicate (devices.rs:443-500, 550-556); state carries across calls."""
        x = np.ascontiguousarray(mono, dtype=np.float32)
        assert x.ndim == 2 and x.shape[0] == self.channels
        out = np.empty((self.channels, n_out, 2), dtype=np.float32)
        used = ctypes.c_int64()
        self._ck(self._L.dspb_resample_dup_stereo(self._h, x.ctypes.data, out.ctypes.data, x.shape[1], n_out, float(target_hz),
                                                  MEM_HOST, None, ctypes.byref(used)))
        return out, used.value

    def process(self, inputs, n_samples: Optional[int] = None) -> List[np.ndarray]:
        """Convenience for tests: numpy in, numpy out, through the host-buffer path."""
        if isinstance(inputs, np.ndarray):
            inputs = [inputs]
        ins = [np.ascontiguousarray(x, dtype=np.float32) for x in inputs]
        n = ins[0].shape[1] if ins else int(n_samples)
        outs = [np.empty((self.channels, n), dtype=np.float32) for _ in range(self._n_out)]
        self.process_host(ins, outs, n)
        return outs

    def node_process(self, node_id: int, port_inputs, n_outputs: int = 1) -> List[np.ndarray]:
        """One SimpleNode::process (node.rs:135-146) on pre-averaged port buffers; None = unconnected."""
        arrs = [None if x is None else np.ascontiguousarray(x, dtype=np.float32) for x in port_inputs]
        n = next(a.shape[1] for a in arrs if a is not None)
        outs = [np.empty((self.channels, n), dtype=np.float32) for _ in range(n_outputs)]
        ip = (ctypes.c_void_p * len(arrs))(*[None if a is None else a.ctypes.data for a in arrs])
        pres = (ctypes.c_uint8 * len(arrs))(*[0 if a is None else 1 for a in arrs])
        op = (ctypes.c_void_p * n_outputs)(*[y.ctypes.data for y in outs])
        self._ck(self._L.dspb_node_process(self._h, node_id, ip, pres, op, n, MEM_HOST, None))
        return outs
