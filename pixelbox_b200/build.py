"""Builds the product library (pixelbox_b200/lib/libpixelbox_b200.so) with nvcc for sm_100a.

In-tree on purpose: the .so is git-ignored but travels with the repo snapshot to the GPU box.
    python -m pixelbox_b200.build [--force] [--verbose]
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
SO = os.path.join(LIBDIR, "libpixelbox_b200.so")
SOURCES = ["api.cu", "range_sort.cu"]
HEADERS = sorted(f for f in os.listdir(CSRC) if f.endswith(".cuh")) + [os.path.join("..", "..", "include", "pixelbox_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-rdc=true", "-DPBX_USE_CDP",          # the exact pass is tail-launched from the finalize kernel
    "-Xcompiler", "-fPIC,-fvisibility=hidden,-O2",
    "-shared",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def needs_build() -> bool:
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return SO
    os.makedirs(LIBDIR, exist_ok=True)
    extra = os.environ.get("PBX_NVCC_EXTRA", "").split()      # experiments only, e.g. -DPBX_EXP_NOMETA
    flags = list(NVCC_FLAGS)
    if os.environ.get("PBX_NO_CDP"):
        # racecheck / synccheck / initcheck of compute-sanitizer do not support CUDA dynamic parallelism: this variant
        # launches the exact pass from the host (always enqueued, returns at once unless a certificate failed)
        flags = [f for f in flags if f not in ("-rdc=true", "-DPBX_USE_CDP")]
    out = os.environ.get("PBX_SO_OUT", SO)
    cmd = [_nvcc()] + flags + extra + (["-Xptxas", "-v"] if verbose else []) + \
          ["-o", out] + [os.path.join(CSRC, s) for s in SOURCES] + ([] if os.environ.get("PBX_NO_CDP") else ["-lcudadevrt"])
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("nvcc failed building libpixelbox_b200.so")
    if verbose:
        sys.stderr.write(res.stderr)
    return SO


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
