"""In-tree build of the C-ABI library (nvcc, sm_100a only).

``python -m smoltts_b200.build`` compiles ``csrc/*.cu`` into
``smoltts_b200/_lib/libsmoltts_b200.so``.  nvcc cross-compiles without a GPU, so this
also runs in the CPU-only build container; the .so is git-ignored but travels to the
GPU box with the repo snapshot.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
LIB_DIR = os.path.join(PKG, "_lib")
LIB_PATH = os.path.join(LIB_DIR, "libsmoltts_b200.so")
STAMP = os.path.join(LIB_DIR, "build.stamp")
SOURCES = ["decode_kernel.cu", "ll2_kernel.cu", "capi.cu", "mimi_kernels.cu", "mimi_encoder.cu", "resample.cu"]
HEADERS = ["common.cuh", "mimi_common.cuh", "dev_model.h", "sampler.cuh", "umma.cuh", "tc_phases.cuh", "tmap_host.h", os.path.join("..", "..", "include", "smoltts_b200.h"),
           os.path.join("..", "..", "include", "smoltts_b200_mimi.h"), os.path.join("..", "..", "include", "smoltts_b200_resample.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC", "-shared",
    "--expt-relaxed-constexpr",
    "-Xptxas", "-v",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (set NVCC=/path/to/nvcc)")


def _digest() -> str:
    h = hashlib.sha256(" ".join(NVCC_FLAGS).encode())
    for name in SOURCES + HEADERS:
        with open(os.path.join(CSRC, name), "rb") as f:
            h.update(name.encode())
            h.update(f.read())
    return h.hexdigest()


def is_current() -> bool:
    if not (os.path.exists(LIB_PATH) and os.path.exists(STAMP)):
        return False
    with open(STAMP) as f:
        return f.read().strip() == _digest()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile the library if sources changed; returns its path."""
    if not force and is_current():
        return LIB_PATH
    os.makedirs(LIB_DIR, exist_ok=True)
    extra = os.environ.get("SMOL_EXTRA_NVCC", "").split()
    cmd = [_nvcc(), *NVCC_FLAGS, *extra, *[os.path.join(CSRC, s) for s in SOURCES], "-o", LIB_PATH, "-lcudart"]
    proc = subprocess.run(cmd, capture_output=True, text=True)
    log = proc.stdout + proc.stderr
    with open(os.path.join(LIB_DIR, "build.log"), "w") as f:
        f.write(" ".join(cmd) + "\n" + log)
    if proc.returncode != 0:
        raise RuntimeError(f"nvcc failed ({proc.returncode}):\n{log[-6000:]}")
    if verbose:
        print(log)
    with open(STAMP, "w") as f:
        f.write(_digest())
    return LIB_PATH


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(path)
