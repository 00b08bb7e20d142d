"""Batched depth-limited minimax on the GPU: the reference's ``OptimalPlayer`` (src/reversi/players/reversi_players.py:
35-77) for thousands of positions in one call, and its ``RandomPlayer`` as depth 0 (``bz_minimax_moves``; the definition
is oracle/minimax_ref.py, the semantics are in include/betazero_b200.h).

    action, value, nodes = best_moves(me, opp, depth=4, size=8, seed=0, keys=game_keys)

``solve`` is the exact endgame solver (``bz_endgame_solve``): the perfect player's move and every move's final disc
difference for positions with at most 20 empty squares.

    action, value, move_value, nodes = solve(me, opp, size=8)
"""
from __future__ import annotations

import torch

from . import _lib, env

MAX_DEPTH = 8  # BZ_MINIMAX_MAX_DEPTH


def check_depth(depth) -> int:
    d = int(depth)
    if not 0 <= d <= MAX_DEPTH:
        raise ValueError(f"minimax depth must be in 0 .. {MAX_DEPTH}; got {depth}")
    return d


def workspace(n: int, device="cuda") -> torch.Tensor:
    """scratch of a bz_minimax_moves call over n roots (torch allocations are 16-byte aligned)"""
    nbytes = int(_lib.load().bz_minimax_workspace_bytes(int(n)))
    return torch.empty(max(nbytes, 16), dtype=torch.uint8, device=device)


def best_moves(me: torch.Tensor, opp: torch.Tensor, depth, size: int = 8, seed: int = 0, keys=0):
    """The minimax move of every mover-relative root (me, opp: int64 CUDA tensors holding uint64 bitboards).

    ``depth``: an int or a tensor of per-root depths in 0 .. 8; ``keys``: the game key of each root (an int or a tensor),
    which with ``seed`` draws the random move when the search returns none (depth 0, or every move worth -inf).
    Returns CUDA tensors (action uint8: row*8 + col, 64 = pass, 255 = game over; value int8: the root's minimax value, the
    disc difference for the mover, +-127 = +-inf; nodes int64: minimax calls of the search)."""
    if size not in (4, 6, 8):
        raise ValueError("size must be 4, 6 or 8 (Reversi)")
    n = me.numel()
    dev = me.device
    if isinstance(depth, torch.Tensor):
        if depth.numel() and not (0 <= int(depth.min()) and int(depth.max()) <= MAX_DEPTH):
            raise ValueError(f"minimax depths must be in 0 .. {MAX_DEPTH}")
        d = depth.to(device=dev, dtype=torch.uint8).contiguous()
    else:
        d = torch.full((n,), check_depth(depth), dtype=torch.uint8, device=dev)
    if isinstance(keys, torch.Tensor):
        k = keys.to(device=dev, dtype=torch.int64).contiguous()
    else:
        k = torch.full((n,), int(keys), dtype=torch.int64, device=dev)
    if d.numel() != n or k.numel() != n or opp.numel() != n:
        raise ValueError("me, opp, depth and keys must have one entry per root")
    action = torch.empty(n, dtype=torch.uint8, device=dev)
    value = torch.empty(n, dtype=torch.int8, device=dev)
    nodes = torch.empty(n, dtype=torch.int64, device=dev)
    ws = workspace(n, dev)
    L = _lib.load()
    _lib.check(L.bz_minimax_moves(_lib.dptr(me.contiguous()), _lib.dptr(opp.contiguous()), _lib.dptr(d), _lib.dptr(k),
                                  int(seed) & (2**64 - 1), n, int(size), _lib.dptr(ws), _lib.dptr(action),
                                  _lib.dptr(value), _lib.dptr(nodes), _lib.stream_ptr()), "bz_minimax_moves")
    return action, value, nodes


SOLVE_MAX_EMPTIES = 20  # BZ_SOLVE_MAX_EMPTIES


def solve(me: torch.Tensor, opp: torch.Tensor, size: int = 8):
    """The exact endgame value of every mover-relative root (me, opp: int64 CUDA tensors holding uint64 bitboards) with
    at most 20 empty squares (``bz_endgame_solve``; the definition is oracle/endgame_ref.py).

    Returns CUDA tensors (action uint8 [n]: the first best move, row*8 + col, 64 = a forced pass, 255 = game over;
    value int8 [n]: the final disc difference for the mover under perfect play, empty squares to nobody; move_value int8
    [n, 65]: the value of every legal move for the mover, the pass at 64, -128 for an action that is not legal; nodes
    int64 [n]: positions the search entered).  ``ValueError`` for a root with more than 20 empties (one device read)."""
    if size not in (4, 6, 8):
        raise ValueError("size must be 4, 6 or 8 (Reversi)")
    n = me.numel()
    if opp.numel() != n:
        raise ValueError("me and opp must have one entry per root")
    dev = me.device
    me, opp = me.contiguous(), opp.contiguous()
    if n:
        _, _, cm, co = env.terminal(me, opp, size)  # the disc counts
        if int((cm.int() + co.int()).min()) < size * size - SOLVE_MAX_EMPTIES:
            raise ValueError(f"the endgame solver takes positions with at most {SOLVE_MAX_EMPTIES} empty squares")
    action = torch.empty(n, dtype=torch.uint8, device=dev)
    value = torch.empty(n, dtype=torch.int8, device=dev)
    move_value = torch.empty((n, 65), dtype=torch.int8, device=dev)
    nodes = torch.empty(n, dtype=torch.int64, device=dev)
    L = _lib.load()
    ws = torch.empty(max(int(L.bz_endgame_workspace_bytes(n)), 16), dtype=torch.uint8, device=dev)
    _lib.check(L.bz_endgame_solve(_lib.dptr(me), _lib.dptr(opp), n, int(size), _lib.dptr(ws), _lib.dptr(action),
                                  _lib.dptr(value), _lib.dptr(move_value), _lib.dptr(nodes), _lib.stream_ptr()),
               "bz_endgame_solve")
    return action, value, move_value, nodes
