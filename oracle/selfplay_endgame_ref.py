"""Sequential restatement of self-play with the endgame handover (``BatchedSelfPlay(endgame_empties=E)``;
bz_selfplay_advance_endgame / bz_selfplay_endgame_play in include/betazero_b200.h).

The game runs mcts_ref.self_play_game's loop -- search, most visited move, record, apply -- until a searched move leaves a
position that is not over and has at most E empty squares (the handover).  From there the perfect player moves: the first
best move of endgame_ref.solve (a forced pass is a pass), recorded with pi = 1/k in float32 on each of the k actions whose
move value equals the root value.  z of every record is the final result for its mover, as before; since play after the
handover is perfect, that is the sign of the handover position's exact value.

``solve(board, player) -> (action, value, move_values)``: ``reference_solver`` runs endgame_ref.solve on the board API;
``c_solver`` runs the C restatement (pyendgame), which is fast enough for 12 empties on 8x8.
"""
from __future__ import annotations

import numpy as np

from . import endgame_ref
from . import mcts_ref as mr

F32 = np.float32


def solver_pi(move_values, value) -> np.ndarray:
    """pi of a solver-played record: 1/k on each of the k actions whose move value is the root value (illegal actions
    hold -128, below any value); one-hot on 64 for a forced pass"""
    mv = np.asarray(move_values, dtype=np.int64)
    opt = mv == int(value)
    pi = np.zeros(65, dtype=np.float32)
    pi[opt] = F32(1) / F32(int(opt.sum()))
    return pi


def reference_solver(board, player):
    a, v, mv, _ = endgame_ref.solve(board, player)
    return a, v, mv


def c_solver(game):
    from . import pyendgame

    def solve(board, player):
        me, opp = game.wire(board, player)
        act, val, mv, _ = pyendgame.endgame_solve(np.array([me], np.uint64), np.array([opp], np.uint64), game.size)
        return int(act[0]), int(val[0]), mv[0].astype(np.int64).tolist()

    return solve


def empties(game, board, player) -> int:
    me, opp = game.wire(board, player)
    return game.size * game.size - bin(me | opp).count("1")


def self_play_game_endgame(game, n_sims: int, c_puct: float, evaluator, endgame_empties: int, solve=reference_solver,
                           max_plies: int = 128, leaves: int = 1, reuse: bool = False, cap_units: int | None = None):
    """One deterministic self-play game with the handover at ``endgame_empties``.  Returns the records (me, opp, player,
    pi float32 [65], action) per ply, the winner (+1 X, -1 O, 0 draw) and the index of the first solver-played record
    (None when the game ended without a handover)."""
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
            cnt, _, _ = m.root_stats()
            a, pi = mr.pick_move(cnt), mr.policy_from_counts(cnt)
        else:
            a, v, mv = solve(board, player)
            pi = solver_pi(mv, v)
        history.append((me, opp, player, pi, a))
        board, player = game.next(board, player, a)
        if handover is None:
            if reuse:
                m.advance(a, board, player, cap_units)
            if (game.terminal_value(board, player) is None and len(history) < max_plies
                    and empties(game, board, player) <= endgame_empties):
                handover = len(history)
    tv = game.terminal_value(board, player)
    winner = 0 if tv is None else int(tv) * player
    return history, winner, handover
