"""Compile the CUDA library in-tree for sm_100a (explicit nvcc; no JIT cache).

    python -m pyperiod_b200.build [--force]

The shared object lands next to this file so it travels with the repo snapshot to the
GPU box; it is git-ignored (history stays source-only).
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_NAME = "libpyperiod_b200.so"
LIB_PATH = os.path.join(HERE, LIB_NAME)
SOURCES = ["pp_periods.cu", "pp_qo.cu", "pp_ramanujan.cu", "pp_extract.cu", "pp_bfreq.cu", "pp_comm.cu", "pp_muresan.cu", "pp_microbench.cu", "pp_long.cu",
           "pp_long_qo.cu", "pp_ram_divisor.cu"]
HEADERS = ["pp_common.cuh", "pp_sweep.cuh", "pp_host.cuh", "pp_chol.cuh", "pp_cg.cuh", "pp_qo.cuh", "pp_long.cuh"]
PUBLIC_HEADER = os.path.join(os.path.dirname(HERE), "include", "pyperiod_b200.h")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared", "-ldl",
    "--threads", "6",          # the translation units compile in parallel
]


def _nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found; cannot build the sm_100a library")
    return exe


def _stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    built = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [PUBLIC_HEADER]
    return any(os.path.getmtime(d) > built for d in deps if os.path.exists(d))


def build(force: bool = False, verbose: bool = False, defines=(), out: str | None = None) -> str:
    """Build libpyperiod_b200.so if missing or older than its sources; return its path.

    `out` names an alternative output file (tuning variants built with `-D...`; load one by
    setting PYPERIOD_B200_LIB)."""
    if out is not None:
        force = True
    if not force and not _stale():
        return LIB_PATH
    cmd = [_nvcc()] + NVCC_FLAGS + [f"-D{d}" for d in defines] + (["-Xptxas", "-v"] if verbose else []) + \
          ["-o", out or LIB_PATH] + [os.path.join(CSRC, s) for s in SOURCES]
    proc = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or proc.returncode != 0:
        sys.stderr.write(proc.stdout + proc.stderr)
    if proc.returncode != 0:
        raise RuntimeError("nvcc failed building " + LIB_NAME)
    return out or LIB_PATH


if __name__ == "__main__":
    outs = [a[6:] for a in sys.argv if a.startswith("--out=")]
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv,
                defines=[a[2:] for a in sys.argv if a.startswith("-D")], out=outs[0] if outs else None))
