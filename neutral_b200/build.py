"""Builds libneutral_b200.so (the C-ABI kernel set) in-tree with nvcc for sm_100a.

``python -m neutral_b200.build`` or :func:`build_library`. The flags are part of the parity
contract: ``-fmad=false`` (no implicit FMA contraction on the device) and
``-ffp-contract=off`` (none on the host side of the same sources); never ``--use_fast_math``.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
# NB200_LIB / NB200_DEFINES build and load an experiment variant next to the product library
# (e.g. NB200_DEFINES=-DNB_HISTORY_MIN_BLOCKS=5 NB200_LIB=libneutral_b200.mb5.so).
LIB = os.path.join(HERE, os.environ.get("NB200_LIB", "libneutral_b200.so"))
SOURCES = ["transport.cu", "stage.cu", "pipeline.cu", "history.cu", "group.cu",
           "tally_batches.cu", "microbench.cu", "capi.cu"]
HEADERS = ["transport.cuh", "nb_device.cuh", "nb_bank.cuh", "nb_math.cuh", "nb_history.cuh",
           "nb_sincos.cuh", "nb_fastmath.cuh", "nb_group.cuh", "nb_nccl_dyn.cuh", "engine.cuh", "glibc_log_table.inc", "glibc_sincos_table.inc",
           os.path.join("..", "..", "include", "neutral_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-fmad=false",
    "-Xcompiler", "-fPIC,-fopenmp,-ffp-contract=off,-O2",
    "-Xptxas", "-v",
]


def find_nvcc() -> str:
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: the b200 kernel set cannot be built")
    return nvcc


def is_stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build_library(force: bool = False, verbose: bool = False) -> str:
    if not force and not is_stale():
        return LIB
    cmd = [find_nvcc()] + NVCC_FLAGS + os.environ.get("NB200_DEFINES", "").split() + ["-shared"] + \
        [os.path.join(CSRC, s) for s in SOURCES] + ["-o", LIB, "-lgomp", "-ldl"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    log = res.stdout + res.stderr
    with open(os.path.join(HERE, "build.log"), "w") as f:
        f.write(" ".join(cmd) + "\n" + log)
    if res.returncode != 0:
        sys.stderr.write(log)
        raise RuntimeError("nvcc failed building libneutral_b200.so")
    if verbose:
        print(log)
    return LIB


if __name__ == "__main__":
    print(build_library(force=True, verbose=True))
