"""Build libparadis_sl.so in-tree with nvcc for sm_100a (no JIT cache, no torch extension)."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_DIR = os.path.join(_HERE, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libparadis_sl.so")
SOURCES = [os.path.join(_HERE, "csrc", "paradis_sl.cu"), os.path.join(_HERE, "csrc", "geo_dwconv.cu")]
HEADERS = [os.path.join(_HERE, "csrc", "sl_device.cuh"), os.path.join(_HERE, "csrc", "sl_sweep.cuh"),
           os.path.join(_HERE, "csrc", "sl_partition.cuh"),
           os.path.join(_HERE, "csrc", "sl_rows.cuh"), os.path.join(_HERE, "csrc", "sl_tangent.cuh"),
           os.path.join(_HERE, "csrc", "sl_f64.cuh"), os.path.join(_HERE, "csrc", "geo_f64.cuh"),
           os.path.join(_HERE, "..", "include", "paradis_sl.h"),
           os.path.join(_HERE, "..", "include", "paradis_sl_tl.h"),
           os.path.join(_HERE, "..", "include", "paradis_sl_bf16.h"),
           os.path.join(_HERE, "..", "include", "paradis_geocyclic.h"),
           os.path.join(_HERE, "..", "include", "paradis_sl_f64.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-shared", "-Xcompiler", "-fPIC"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; libparadis_sl.so cannot be built")


def is_stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(s) > t for s in SOURCES + HEADERS if os.path.exists(s))


def build_library(force: bool = False, verbose: bool = False) -> str:
    if not force and not is_stale():
        return LIB_PATH
    os.makedirs(LIB_DIR, exist_ok=True)
    cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB_PATH] + SOURCES
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return LIB_PATH


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
