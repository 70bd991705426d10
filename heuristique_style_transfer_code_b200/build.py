"""Builds csrc/libgramhead.so for sm_100a with nvcc (no torch headers, no JIT cache: the .so stays in-tree)."""
from __future__ import annotations

import os
import shutil
import subprocess

CSRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc")
LIB_PATH = os.path.join(CSRC, "libgramhead.so")
SOURCES = ["gramhead.cu", "common.cuh", "gram_fwd.cuh", "pair.cuh", "gram_fwd_pair.cuh", "gram_bwd2.cuh", "gram_bwd_pair.cuh",
           "umma_gemm.cuh", "tgemm_pair.cuh", "launch.cuh", "attn_head.cuh", "attn_head2.cuh", "preprocess.cuh", "transpose.cuh", "patchgan.cuh", "pool.cuh", "stem.cuh", "style_loss.cuh"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.isfile(cand):
            return cand
    raise RuntimeError("gramhead: nvcc not found (set NVCC=/path/to/nvcc)")


def is_stale() -> bool:
    if not os.path.isfile(LIB_PATH):
        return True
    built = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, s) for s in SOURCES]
    deps.append(os.path.join(os.path.dirname(os.path.dirname(CSRC)), "include", "gramhead.h"))
    return any(os.path.getmtime(d) > built for d in deps if os.path.isfile(d))


def build_library(force: bool = False, verbose: bool = False) -> str:
    if not force and not is_stale():
        return LIB_PATH
    cmd = [_nvcc(), *NVCC_FLAGS, "gramhead.cu", "-o", LIB_PATH + ".tmp"]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    res = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("gramhead: nvcc failed\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    os.replace(LIB_PATH + ".tmp", LIB_PATH)
    return LIB_PATH


if __name__ == "__main__":
    print(build_library(force=True, verbose=True))
