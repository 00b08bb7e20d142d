"""Builds libbetazero_b200.so (the C-ABI CUDA library) in-tree for sm_100a.

    python -m betazero_b200.build [--force]

The .so is git-ignored but travels to the GPU box with the gpurun snapshot.
"""
from __future__ import annotations

import fcntl
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libbetazero_b200.so")
SOURCES = ("env.cu", "mcts.cu", "selfplay.cu", "mlp_pair.cu", "mlp_pair2.cu", "minimax.cu")
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "--fmad=false",  # PUCT arithmetic must round op by op (bit-exact visit counts); intrinsics enforce it too
    "-Xcompiler", "-fPIC", "-shared",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the CUDA extension cannot be built (there is no CPU fallback)")


def sources():
    return [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


STAMP = LIB + ".srchash"  # hash of the sources the library was built from (travels with the .so, like it git-ignored)


def _deps():
    return sorted([os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "betazero_b200.h")])


def source_hash() -> str:
    """Content hash of every source the library depends on (+ the compiler flags).  Staleness is decided by CONTENT,
    not by mtimes: a snapshot copied to another box does not keep file times, and a rebuild started by every rank of a
    torchrun job at once is exactly the race this avoids."""
    h = hashlib.sha256(" ".join(NVCC_FLAGS + list(SOURCES)).encode())
    for d in _deps():
        h.update(os.path.basename(d).encode())
        with open(d, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def needs_build() -> bool:
    if not os.path.exists(LIB) or not os.path.exists(STAMP):
        return True
    try:
        return open(STAMP).read().strip() != source_hash()
    except OSError:
        return True


def build(force: bool = False, verbose: bool = False) -> str:
    """Build under an inter-process lock, into a temporary file that is renamed over the library: concurrent ranks
    either find a complete, current library or wait for the one rank that is building it."""
    if not force and not needs_build():
        return LIB
    with open(LIB + ".lock", "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not needs_build():  # another process built it while we waited
                return LIB
            tmp = f"{LIB}.tmp.{os.getpid()}"
            cmd = [_nvcc(), *NVCC_FLAGS, "-o", tmp, *sources()]
            if verbose:
                cmd.insert(1, "-Xptxas")
                cmd.insert(2, "-v")
                print(" ".join(cmd))
            try:
                subprocess.check_call(cmd)
                os.replace(tmp, LIB)
            finally:
                if os.path.exists(tmp):
                    os.remove(tmp)
            with open(STAMP + ".tmp", "w") as f:
                f.write(source_hash())
            os.replace(STAMP + ".tmp", STAMP)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
