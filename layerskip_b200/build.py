"""Build liblsk.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

`python -m layerskip_b200.build` or `__graft_entry__.build()`.  nvcc cross-compiles without a
GPU; the resulting .so is git-ignored but travels to the GPU box with the gpurun snapshot.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.path.join(PKG_DIR, "liblsk.so")
STAMP_PATH = os.path.join(PKG_DIR, ".liblsk.stamp")
INCLUDE_DIR = os.path.join(os.path.dirname(PKG_DIR), "include")
SOURCES = ["engine.cu"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "--shared", "-Xcompiler", "-fPIC",
]


def _digest_inputs() -> list:
    """Every file the library is compiled from: all of csrc/ (engine.cu includes the headers,
    so a new header needs no list to be kept in step) and the public C header."""
    files = [os.path.join(CSRC, n) for n in sorted(os.listdir(CSRC))]
    files.append(os.path.join(INCLUDE_DIR, "lsk.h"))
    return [p for p in files if os.path.isfile(p)]


def _digest() -> str:
    h = hashlib.sha256()
    for path in _digest_inputs():
        h.update(os.path.basename(path).encode() + b"\0")
        with open(path, "rb") as f:
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def needs_build() -> bool:
    if not os.path.exists(LIB_PATH) or not os.path.exists(STAMP_PATH):
        return True
    with open(STAMP_PATH) as f:
        return f.read().strip() != _digest()


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB_PATH
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: cannot build liblsk.so")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + \
          ["-o", LIB_PATH] + [os.path.join(CSRC, s) for s in SOURCES] + ["-lnccl"]
    proc = subprocess.run(cmd, capture_output=True, text=True)
    if verbose:
        sys.stderr.write(proc.stderr)
    if proc.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + proc.stdout + proc.stderr)
    with open(STAMP_PATH, "w") as f:
        f.write(_digest())
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
