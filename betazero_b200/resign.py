"""Resignation in self-play: which games are audited, the false-positive rate of a threshold, and its calibration.

Definition (oracle/selfplay_resign_ref.py, include/betazero_b200.h bz_selfplay_resign_state): a searched ply's q is
W / N of its most visited root edge from the mover's point of view; a game that is not audited resigns at its first
searched ply with q < threshold, and its mover loses.  Game g is audited iff philox_u32(seed, g, 0xFFFFFFFF) <
floor(fraction * 2^32); audited games never resign, so they show what resigning would have cost:

- the would-be resigner of an audited game for a threshold v is its first record r (ply order) with q_r < v; the game
  is a FALSE POSITIVE iff it has one and z_r >= 0 (the side that would have resigned drew or won);
- FP(v) = false positives / audited games;
- ``calibrate(records, target)`` is the largest v among {-1} and the audited records' q such that FP(u) <= target for
  every such candidate u <= v (FP is not monotone in v; the prefix keeps the answer well defined).

``records`` is a dict of equal-length arrays (numpy, or tensors on any device) as ``BatchedSelfPlay.drain_replay`` and
``dist.gather_replay`` return them: "game", "ply", "q", "z", plus a per-record bool "audited" (``with_audit``).
"""
from __future__ import annotations

import math

import numpy as np

AUDIT_COUNTER = 0xFFFFFFFF  # the Philox counter of the audit draw: never a ply


def audit_below(fraction: float) -> int:
    """floor(fraction * 2^32): the bz_selfplay_resign_state field for an audited fraction in [0, 1]"""
    f = float(fraction)
    if not 0.0 <= f <= 1.0:
        raise ValueError(f"resign_audit must be a fraction in [0, 1]; got {fraction}")
    return int(math.floor(f * 2.0 ** 32))


def check_threshold(v) -> float:
    """a threshold in [-1, 1] (-1 never resigns), as float32"""
    t = float(np.float32(v))
    if not -1.0 <= t <= 1.0:  # NaN fails too
        raise ValueError(f"resign threshold must be in [-1, 1]; got {v}")
    return t


def audited(game_ids, seed: int, fraction: float):
    """bool per game id (a CUDA tensor, on its device): philox_u32(seed, g, 0xFFFFFFFF) < floor(fraction * 2^32)"""
    import torch

    from . import _lib

    below = audit_below(fraction)
    g = game_ids.to(torch.int64).contiguous()
    n = g.numel()
    ply = torch.full((n,), -1, dtype=torch.int32, device=g.device)  # uint32 0xFFFFFFFF
    u = torch.empty(n, dtype=torch.int32, device=g.device)
    if n:
        _lib.check(_lib.load().bz_philox_u32(int(seed), _lib.dptr(g), _lib.dptr(ply), _lib.dptr(u), n, _lib.stream_ptr()),
                   "bz_philox_u32")
    return (u.to(torch.int64) & 0xFFFFFFFF) < below


def with_audit(records: dict, seed: int, fraction: float) -> dict:
    """``records`` plus the per-record "audited" flag of its game"""
    out = dict(records)
    out["audited"] = audited(records["game"], seed, fraction)
    return out


def _np(x):
    return x.cpu().numpy() if hasattr(x, "cpu") else np.asarray(x)


def _audited_games(records: dict):
    """per audited game, in game order: (q float32, z int) of its records in ply order"""
    game, ply = _np(records["game"]).astype(np.int64), _np(records["ply"]).astype(np.int64)
    q, z, aud = _np(records["q"]).astype(np.float32), _np(records["z"]).astype(np.int64), _np(records["audited"]).astype(bool)
    idx = np.flatnonzero(aud)
    idx = idx[np.lexsort((ply[idx], game[idx]))]
    bounds = np.flatnonzero(np.diff(game[idx])) + 1
    return [(q[i], z[i]) for i in np.split(idx, bounds) if i.size]


def audited_games(records: dict) -> int:
    """the number of audited games in ``records``"""
    return len(_audited_games(records))


def _low_intervals(games):
    """For each game, its would-be resigner is record i_j for thresholds v in (l_j, l_{j-1}], where i_1 < i_2 < ... are
    the records that set a new running minimum l_1 > l_2 > ... of q (NaN never resigns; l_0 = +inf).  Returns the
    (l_j, l_{j-1}) bounds of the records with z >= 0: the thresholds at which the game is a false positive."""
    lo, hi = [], []
    for q, z in games:
        qe = np.where(np.isnan(q), np.float32(np.inf), q)
        prev = np.concatenate(([np.float32(np.inf)], np.minimum.accumulate(qe)[:-1]))
        new = np.flatnonzero(qe < prev)
        for i in new:
            if z[i] >= 0:
                lo.append(qe[i])
                hi.append(prev[i])
    return np.asarray(lo, np.float32), np.asarray(hi, np.float32)


def false_positive_rate(records: dict, v: float) -> float:
    """FP(v) over the audited games of ``records``; 0.0 without audited games"""
    games = _audited_games(records)
    if not games:
        return 0.0
    v = np.float32(v)
    lo, hi = _low_intervals(games)
    return int(np.count_nonzero((lo < v) & (v <= hi))) / len(games)


def calibrate(records: dict, target: float, keep: float = -1.0) -> float:
    """the largest candidate v (-1 or an audited record's q) with FP(u) <= target for every candidate u <= v; ``keep``
    when ``records`` has no audited game"""
    if not target >= 0.0:
        raise ValueError(f"the false-positive target must be >= 0; got {target}")
    games = _audited_games(records)
    if not games:
        return float(keep)
    qs = np.concatenate([q for q, _ in games])
    cands = np.unique(np.concatenate(([np.float32(-1)], qs[~np.isnan(qs)])).astype(np.float32))
    lo, hi = _low_intervals(games)
    # the false positives at candidate c: intervals (lo, hi] that hold c, counted with a difference array
    diff = np.zeros(cands.size + 1, np.int64)
    np.add.at(diff, np.searchsorted(cands, lo, side="right"), 1)
    np.add.at(diff, np.searchsorted(cands, hi, side="right"), -1)
    fp = np.cumsum(diff[:-1])
    bad = np.flatnonzero(fp / len(games) > target)
    k = int(bad[0]) if bad.size else cands.size
    return float(cands[k - 1]) if k > 0 else -1.0
