"""Sequential restatement of self-play with resignation (``BatchedSelfPlay(resign_threshold=v, resign_audit=f)``;
bz_selfplay_advance_resign / bz_selfplay_endgame_play_resign in include/betazero_b200.h).

After a ply's search the root's edges hold (N, W) from the mover's point of view (mcts_ref.MCTS.expand_backup negates
the value before it adds it to the edge into a node).

- q of a searched ply: a* is the most visited root action, lowest action id on ties (the greedy pick, also on plies that
  sample the move); q = float32(W[a*]) / float32(N[a*]), one correctly rounded division.  A root with no visits has
  q = NaN and never resigns.  (Not the root's mean sum W / sum N: no fixed float32 summation order would pin it.)
- Audited games: game g is audited iff philox_u32(seed, g, 0xFFFFFFFF) < audit_below, audit_below = floor(fraction *
  2^32) in 0 .. 2^32 (fraction 1 audits every game).  The counter 0xFFFFFFFF is never a ply, so the draw is independent
  of move sampling.  An audited game never resigns.
- Resignation: a searched ply of a game that is not audited resigns iff q < threshold (float32 compare; threshold in
  [-1, 1], -1 never fires).  The position is recorded as always (board, pi from the visit counts, the picked action), the
  mover loses (winner = -player), the game is flushed like a finished game (z = winner * player for every record) and
  the slot restarts; the move is not played.  The check comes before the move is applied, so before the endgame
  handover test of the same ply.  Solver-played plies never resign and carry q = NaN.
- False positives: among the audited games of a set of finished games, for a threshold v a game's would-be resigner is
  its first record r (ply order) with q_r < v; the game is a false positive iff it has one and z_r >= 0 (the side that
  would have resigned drew or won).  FP(v) = false positives / audited games.
- Calibration: calibrate(games, target) is the largest v among {-1} and the q of the audited records such that
  FP(u) <= target for every such candidate u <= v (a prefix: FP is not monotone in v, the answer is still well
  defined).  With no audited games the threshold is kept.
"""
from __future__ import annotations

import math

import numpy as np

from . import mcts_ref as mr
from . import selfplay_endgame_ref as ser
from .minimax_ref import philox_u32

F32 = np.float32
NAN = F32("nan")
AUDIT_COUNTER = 0xFFFFFFFF


def audit_below(fraction: float) -> int:
    """floor(fraction * 2^32) for fraction in [0, 1]"""
    return int(math.floor(float(fraction) * 2.0 ** 32))


def audited(seed: int, game_id: int, below: int) -> bool:
    return philox_u32(seed, game_id, AUDIT_COUNTER) < below


def root_q(counts, W) -> np.float32:
    """q of a searched ply from mcts_ref.MCTS.root_stats' (counts, W)"""
    counts = np.asarray(counts)
    if int(counts.sum()) == 0:
        return NAN
    a = mr.pick_move(counts)
    return F32(W[a]) / F32(int(counts[a]))


def self_play_game_resign(game, n_sims: int, c_puct: float, evaluator, threshold: float, is_audited: bool = False,
                          endgame_empties: int = 0, solve=ser.reference_solver, max_plies: int = 128, leaves: int = 1,
                          reuse: bool = False, cap_units: int | None = None):
    """One deterministic self-play game with resignation (and the endgame handover at ``endgame_empties`` > 0, as in
    selfplay_endgame_ref).  Returns the records (me, opp, player, pi float32 [65], action, q float32) per ply, the
    winner (+1 X, -1 O, 0 draw), the index of the first solver-played record (None without a handover) and whether the
    game resigned (its last record is then the resigning ply)."""
    v = F32(threshold)
    board, player = game.initial()
    history, m, handover = [], None, None
    while game.terminal_value(board, player) is None and len(history) < max_plies:
        me, opp = game.wire(board, player)
        if handover is None:
            if m is None or not reuse:
                m = mr.MCTS(game, c_puct, evaluator)
                m.reset(board, player)
            if leaves > 1:
                m.run_vl(n_sims, leaves)
            else:
                m.run(n_sims)
            cnt, W, _ = m.root_stats()
            a, pi, q = mr.pick_move(cnt), mr.policy_from_counts(cnt), root_q(cnt, W)
        else:
            a, val, mv = solve(board, player)
            pi, q = ser.solver_pi(mv, val), NAN
        history.append((me, opp, player, pi, a, q))
        if handover is None and not is_audited and q < v:
            return history, -player, handover, True
        board, player = game.next(board, player, a)
        if handover is None:
            if reuse:
                m.advance(a, board, player, cap_units)
            if (endgame_empties and game.terminal_value(board, player) is None and len(history) < max_plies
                    and ser.empties(game, board, player) <= endgame_empties):
                handover = len(history)
    tv = game.terminal_value(board, player)
    winner = 0 if tv is None else int(tv) * player
    return history, winner, handover, False


def false_positive_rate(games, v: float) -> float:
    """FP(v) over ``games``: a list of (q, z) per AUDITED game, records in ply order; 0 without games"""
    if not games:
        return 0.0
    v = F32(v)
    fp = 0
    for q, z in games:
        for r in range(len(q)):
            if F32(q[r]) < v:
                fp += int(z[r]) >= 0
                break
    return fp / len(games)


def calibrate(games, target: float, keep: float) -> float:
    """the largest candidate v with FP(u) <= target for every candidate u <= v; ``keep`` without audited games"""
    if not games:
        return keep
    cands = sorted({F32(-1)} | {F32(x) for q, _ in games for x in q if not np.isnan(x)})
    best = F32(-1)
    for u in cands:
        if false_positive_rate(games, u) > target:
            break
        best = u
    return float(best)
