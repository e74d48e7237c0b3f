"""Builds libpcb200.so (hand-written sm_100a CUDA behind the C ABI of include/pcb200.h) in-tree with nvcc.

    python -m pointcontrast_b200.build [--force]

The .so is git-ignored but travels to the GPU box with the gpurun snapshot.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SOURCES = ["coords.cu", "voxel.cu", "conv.cu", "conv_tc5.cu", "bn.cu", "loss.cu", "nce_tc5.cu", "unit.cu", "seg_eval.cu"]
OUT = os.path.join(HERE, "libpcb200.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "--threads", "4",
         "-Xcompiler", "-fPIC", "-shared", "-cudart", "static"]


def _stale():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "pcb200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not _stale():
        return OUT
    cmd = [NVCC] + FLAGS + [os.path.join(CSRC, s) for s in SOURCES] + ["-o", OUT]
    if verbose:
        print(" ".join(cmd))
    subprocess.run(cmd, check=True)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
