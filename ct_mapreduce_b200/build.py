"""Builds libctmr.so (hand-written sm_100a kernels + C ABI) in-tree with nvcc.

    python -m ct_mapreduce_b200.build [--force] [--verbose]

nvcc cross-compiles for sm_100a without a GPU; the .so lands next to this file so that it
travels to the GPU box with the repository snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libctmr.so")
SOURCES = ["ctmr_map.cu", "ctmr_reduce.cu", "ctmr_api.cu", "ctmr_pipeline.cu", "ctmr_frontend.cu", "ctmr_frontend_api.cu", "ctmr_sets.cu", "ctmr_synth_kernels.cu", "ctmr_synth_pages.cu"]
# measured-and-rejected K_map variants (v1 global-memory walk, dynamic scheduling, TMA bulk loader): only with CTMR_EXPERIMENTS=1
EXPERIMENT_SOURCES = ["ctmr_map_alt.cu"]
DEPS = SOURCES + EXPERIMENT_SOURCES + ["ctmr_ctx.cuh", "ctmr_kernels.cuh", "ctmr_common.cuh", "ctmr_stream.cuh", "ctmr_device.cuh", "ctmr_synth.h",
                  "ctmr_synth_ecpoints.inc",
                  os.path.join("..", "..", "include", "ctmr.h"), os.path.join("..", "..", "include", "ctmr_frontend.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC",
    "--expt-relaxed-constexpr",
    "-shared",
]


def _nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libctmr.so must be built where the CUDA toolkit is installed")


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, d)) > t for d in DEPS) or os.path.getmtime(__file__) > t


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    exp = os.environ.get("CTMR_EXPERIMENTS", "0") == "1"
    cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + (["-DCTMR_EXPERIMENTS=1"] if exp else []) + \
          [os.path.join(CSRC, s) for s in SOURCES + (EXPERIMENT_SOURCES if exp else [])] + ["-o", LIB + ".tmp", "-lcudart"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or r.returncode:
        sys.stderr.write(r.stdout + r.stderr)
    if r.returncode:
        raise RuntimeError("nvcc failed building libctmr.so")
    os.replace(LIB + ".tmp", LIB)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
