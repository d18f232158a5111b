"""Builds libmpcb200.so (hand-written CUDA for sm_100a + the C ABI) in-tree with nvcc.

    python -m diplomjourney_b200.build [--force]

nvcc cross-compiles without a GPU; the .so is git-ignored but travels with the tree.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.environ.get("MPCB_LIB") or os.path.join(HERE, "lib", "libmpcb200.so")   # MPCB_LIB: developer override
SOURCES = ["mpcb_kernels.cu", "mpcb_loop.cu", "mpcb_api.cu", "mpcb_nccl.cu"]
HEADERS = ["mpcb_types.cuh", "mpcb_bounds.cuh", "mpcb_exact.cuh", "mpcb_handle.cuh", "mpcb_events.cuh", "mpcb_noise.cuh", "mpcb_pcg64.cuh", "mpcb_screen.cuh", os.path.join("..", "..", "include", "mpcb200.h")]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "--shared",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the CUDA library cannot be built (there is no CPU fallback)")


def source_hash() -> str:
    """Hash of everything the library is built from (sources, headers, flags): what decides staleness.  mtimes do
    not survive a copy of the tree to another box; contents do."""
    h = hashlib.sha256(" ".join(NVCC_FLAGS).encode())
    for name in SOURCES + HEADERS:
        with open(os.path.join(CSRC, name), "rb") as f:
            h.update(name.encode() + b"\0" + f.read())
    return h.hexdigest()


def needs_build(lib: str | None = None) -> bool:
    lib = lib or LIB
    try:
        with open(lib + ".srchash") as f:
            return not os.path.exists(lib) or f.read().strip() != source_hash()
    except OSError:
        return True


def build_library(force: bool = False, verbose: bool = False, extra_flags=(), out: str | None = None) -> str:
    """Compiles the library with nvcc unless the one on disk was built from these very sources (force=True: always).
    A library named by MPCB_LIB is a developer's variant and is used as it is."""
    out = out or LIB
    if not force and out == LIB and (os.environ.get("MPCB_LIB") or not needs_build()):
        if not os.path.exists(LIB):
            raise RuntimeError(f"MPCB_LIB={LIB} does not exist")
        return LIB
    os.makedirs(os.path.dirname(out), exist_ok=True)
    cmd = [_nvcc()] + NVCC_FLAGS + list(extra_flags) + (["-Xptxas", "-v"] if verbose else []) + \
          [os.path.join(CSRC, s) for s in SOURCES] + ["-o", out, "-ldl"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + r.stdout + r.stderr)
    if not extra_flags:
        with open(out + ".srchash", "w") as f:
            f.write(source_hash() + "\n")
    if verbose:
        print(r.stderr)
    return out


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
