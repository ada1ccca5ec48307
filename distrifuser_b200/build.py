"""Builds libdistrifuser_b200.so (hand-written sm_100a CUDA behind the C ABI of include/distrifuser_b200.h).

In-tree build so the .so travels with the repo snapshot to the GPU box; nvcc cross-compiles without a GPU."""
from __future__ import annotations

import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libdistrifuser_b200.so")
SOURCES = ("comm.cu", "groupnorm.cu", "halo.cu", "attention.cu", "elementwise.cu", "linear.cu", "allreduce.cu")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
         "-Xcompiler", "-fPIC", "-shared"]


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "distrifuser_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False, out: str | None = None, csrc: str | None = None) -> str:
    """`out` / `csrc`: build a variant (DF_NVCC_FLAGS, another source tree) next to the shipped library for A/B runs (DF_LIB_PATH)."""
    if out or csrc:
        force = True
    if not force and not _stale():
        return LIB
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: cannot build libdistrifuser_b200.so")
    extra = os.environ.get("DF_NVCC_FLAGS", "").split()          # e.g. -DDF_EMU_PAIRS_OF_8=0 for kernel experiments
    cmd = [nvcc, *FLAGS, *extra, "-I", os.path.join(HERE, "..", "include"), "-o", out or LIB, *[os.path.join(csrc or CSRC, s) for s in SOURCES]]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + r.stdout + r.stderr)
    if verbose:
        print(r.stderr)
    return out or LIB


if __name__ == "__main__":
    print(build(force=True, verbose=True))
