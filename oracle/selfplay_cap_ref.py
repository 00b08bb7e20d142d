"""Sequential restatement of self-play with randomized search budgets (``BatchedSelfPlay(fast_sims=n, full_fraction=p)``;
bz_selfplay_cap_layout / bz_selfplay_advance_cap / bz_selfplay_endgame_play_cap in include/betazero_b200.h).  KataGo's
playout cap randomization (Wu, arXiv:1902.10565): full searches give the policy targets, cheap ones move the games on.

- Draw: a ply of game g at ply index t (the t that keys move sampling) is full iff philox_u32(seed, g, 0x80000000 | t)
  < full_below, full_below = floor(p * 2^32) in 0 .. 2^32 (p = 1: every ply is full).  The counter is never a ply
  (t < 128) and never the resignation audit's 0xFFFFFFFF, so the draw is independent of both.
- Search: a full ply is searched with n_sims simulations, a fast ply with fast_sims (2 K <= fast_sims <= n_sims, K the
  leaves per iteration); both from a fresh tree with the same net.  Root noise, when it is on, applies to full plies
  only.  The move rule is the same for both: sampled ~ N for ply < temp_plies (Philox keyed by (seed, g, ply): the first
  action, in ascending id, whose inclusive prefix sum of N exceeds floor(u32 * sum N / 2^32)), the most visited action
  (lowest id on ties) after.
- Records: every ply is recorded as without the option (board, pi from the visit counts, action, and q of
  selfplay_resign_ref), plus full (1 or 0).  Solver-played plies after an endgame handover are full: they are exact labels.
  Training uses the full records; fast records keep their game's z.
- Composition: resignation is tested at every searched ply, full or fast; the endgame handover is unchanged.
- Identities: p = 1 gives the games without the option with every flag 1; fast_sims == n_sims gives those games with
  the flags of the draw.

``search(board, player, n) -> (counts [65], W [65])``: the search of one fresh tree; the default runs mcts_ref.MCTS with
``evaluator`` (MCTS.run, or MCTS.run_vl with ``leaves`` > 1).  The GPU tests plug in a single-tree
bz_mcts_search_fused, which a tree of the batched search equals bit for bit.
"""
from __future__ import annotations

import math

import numpy as np

from . import mcts_ref as mr
from . import selfplay_endgame_ref as ser
from . import selfplay_resign_ref as srr
from .minimax_ref import philox_u32

FULL_COUNTER = 0x80000000


def full_below(fraction: float) -> int:
    """floor(fraction * 2^32) for fraction in [0, 1]"""
    return int(math.floor(float(fraction) * 2.0 ** 32))


def is_full(seed: int, game_id: int, ply: int, below: int) -> bool:
    return philox_u32(seed, game_id, FULL_COUNTER | int(ply)) < below


def sampled_move(counts, seed: int, game_id: int, ply: int) -> int:
    """the move sampled ~ N (bz_selfplay_advance): the first action whose inclusive prefix sum exceeds
    floor(philox_u32(seed, g, ply) * sum N / 2^32)"""
    counts = np.asarray(counts, dtype=np.int64)
    target = (philox_u32(seed, game_id, ply) * int(counts.sum())) >> 32
    return int(np.flatnonzero(np.cumsum(counts) > target)[0])


def mcts_search(game, c_puct: float, evaluator, leaves: int = 1):
    def search(board, player, n):
        m = mr.MCTS(game, c_puct, evaluator)
        m.reset(board, player)
        if leaves > 1:
            m.run_vl(n, leaves)
        else:
            m.run(n)
        cnt, W, _ = m.root_stats()
        return cnt, W

    return search


def self_play_game_cap(game, n_sims: int, fast_sims: int, search, seed: int, game_id: int, below: int,
                       temp_plies: int = 0, threshold: float | None = None, is_audited: bool = False,
                       endgame_empties: int = 0, solve=ser.reference_solver, max_plies: int = 128):
    """One self-play game (id ``game_id``) with randomized budgets, resignation at ``threshold`` (None: off) and the endgame
    handover at ``endgame_empties`` > 0.  Returns the records (me, opp, player, pi float32 [65], action, q float32, full)
    per ply, the winner (+1 X, -1 O, 0 draw), the index of the first solver-played record (None without a handover) and
    whether the game resigned."""
    v = srr.NAN if threshold is None else np.float32(threshold)
    board, player = game.initial()
    history, handover = [], None
    while game.terminal_value(board, player) is None and len(history) < max_plies:
        me, opp = game.wire(board, player)
        t = len(history)
        if handover is None:
            full = is_full(seed, game_id, t, below)
            cnt, W = search(board, player, n_sims if full else fast_sims)
            cnt = np.asarray(cnt)
            a = sampled_move(cnt, seed, game_id, t) if t < temp_plies and cnt.sum() > 0 else mr.pick_move(cnt)
            pi, q = mr.policy_from_counts(cnt), srr.root_q(cnt, W)
        else:
            a, val, mv = solve(board, player)
            pi, q, full = ser.solver_pi(mv, val), srr.NAN, True
        history.append((me, opp, player, pi, a, q, int(full)))
        if handover is None and not is_audited and q < v:
            return history, -player, handover, True
        board, player = game.next(board, player, a)
        if (handover is None and endgame_empties and game.terminal_value(board, player) is None
                and len(history) < max_plies and ser.empties(game, board, player) <= endgame_empties):
            handover = len(history)
    tv = game.terminal_value(board, player)
    winner = 0 if tv is None else int(tv) * player
    return history, winner, handover, False
