"""TEST INFRASTRUCTURE ONLY -- ctypes front end of oracle/libendgame.so (endgame.c, which includes minimax.c's rules),
the C restatement of the endgame definition (endgame_ref.py) without pruning: the checker of bz_endgame_solve.  Built
with gcc on first use, like pyminimax's library (content hash of both sources beside the library, inter-process
lock)."""
from __future__ import annotations

import ctypes as C
import fcntl
import hashlib
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "endgame.c")
_SOURCES = (_SRC, os.path.join(_HERE, "minimax.c"))
_SO = os.path.join(_HERE, "libendgame.so")
_CFLAGS = ["-O2", "-fPIC", "-shared", "-fopenmp", "-Wall", "-Wextra", "-std=c11"]
_lib = None


def _src_hash() -> str:
    h = hashlib.sha256(" ".join(_CFLAGS).encode())
    for path in _SOURCES:
        with open(path, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def build(force: bool = False) -> str:
    stamp = _SO + ".srchash"

    def stale():
        try:
            return not os.path.exists(_SO) or open(stamp).read().strip() != _src_hash()
        except OSError:
            return True

    if not force and not stale():
        return _SO
    with open(_SO + ".lock", "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if force or stale():
                tmp = f"{_SO}.tmp.{os.getpid()}"
                subprocess.check_call(["gcc", *_CFLAGS, "-o", tmp, _SRC])
                os.replace(tmp, _SO)
                with open(stamp + ".tmp", "w") as f:
                    f.write(_src_hash())
                os.replace(stamp + ".tmp", stamp)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return _SO


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_SO)
        p = C.c_void_p
        L.orc_endgame_solve.argtypes = [p, p, C.c_int64, C.c_int, p, p, p, p]
        L.orc_endgame_solve.restype = None
        _lib = L
    return _lib


def endgame_solve(me, opp, size: int = 8):
    """plain negamax of every root to the end of the game (bz_endgame_solve's semantics):
    (action uint8 [n], value int8 [n], move_value int8 [n, 65], nodes int64 [n])"""
    me, opp = np.ascontiguousarray(me, np.uint64), np.ascontiguousarray(opp, np.uint64)
    n = me.size
    act, val, mv, nodes = np.empty(n, np.uint8), np.empty(n, np.int8), np.empty((n, 65), np.int8), np.empty(n, np.int64)
    lib().orc_endgame_solve(me.ctypes.data, opp.ctypes.data, n, int(size), act.ctypes.data, val.ctypes.data,
                            mv.ctypes.data, nodes.ctypes.data)
    return act, val, mv, nodes
