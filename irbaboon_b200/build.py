"""Build libirb_b200.so (CUDA kernels + C ABI) in-tree with nvcc for sm_100a.

The shared object is git-ignored but travels to the GPU box with the gpurun snapshot.  Rebuilds only when a
source is newer than the library.  Usage: ``python -m irbaboon_b200.build [--force] [--verbose]``.
"""
import os
import subprocess
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
CSRC = os.path.join(_HERE, "csrc")
LIB = os.path.join(_HERE, "libirb_b200.so")
SOURCES = ["irb_engine.cu", "irb_spectral.cu", "irb_benchaids.cu"]
HEADERS = ["irb_chop.cuh", "irb_fft.cuh", "irb_ir_load.cuh", "irb_kernels.cuh", "irb_mac_p.cuh", "irb_mac_mx.cuh", "irb_spectral.cuh", "irb_common.hpp", "irb_tuning.hpp",
           os.path.join(_ROOT, "include", "irb_b200.h"), os.path.join(_ROOT, "include", "irb_b200_bench.h")]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC", "-shared", "-t", "3",
]


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + [h if os.path.isabs(h) else os.path.join(CSRC, h) for h in HEADERS]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not _stale():
        return LIB
    cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES]
    subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
