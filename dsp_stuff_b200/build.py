"""Builds libdspb200.so (CUDA kernels + C ABI) in-tree for sm_100a.  `python -m dsp_stuff_b200.build`."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libdspb200.so")
DRIVER = os.path.join(HERE, "dspb_run")
SOURCES = ["engine.cpp", "fused_chain.cu", "fir.cu", "fir_fft.cu", "fir_toeplitz.cu", "boundary.cu", "reset.cu"]
HEADERS = ["plan.h", "json_min.h", "exact_math.cuh", "dspb_run.cpp", os.path.join("..", "..", "include", "dspb200.h")]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]


def _nvcc() -> str:
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    raise RuntimeError("nvcc not found")


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    objs = []
    bdir = os.path.join(HERE, "build")
    os.makedirs(bdir, exist_ok=True)
    common = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-I", os.path.join(HERE, "..", "include")] + ARCH
    for src in SOURCES:
        obj = os.path.join(bdir, os.path.splitext(src)[0] + ".o")
        cmd = [_nvcc()] + common + ["-c", os.path.join(CSRC, src), "-o", obj]
        if src == "fused_chain.cu":
            # -fmad=false: belt and braces, parity-critical arithmetic also uses *_rn intrinsics
            cmd += ["-fmad=false", "-diag-suppress", "177"]  # 177: unused `rec` members of chains the ws kernel never takes
        if verbose:
            cmd += ["-Xptxas", "-v"]
            print(" ".join(cmd))
        subprocess.check_call(cmd)
        objs.append(obj)
    subprocess.check_call([_nvcc(), "-shared", "-o", LIB] + objs + ARCH + ["-cudart", "static"])
    # headless C++ driver over the C ABI (links the shared library only)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-o", DRIVER, os.path.join(CSRC, "dspb_run.cpp"), "-L", HERE,
                           "-ldspb200", "-Wl,-rpath,$ORIGIN"])
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
