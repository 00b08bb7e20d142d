"""The win/draw/loss endgame result of bz_endgame_solve_wld (include/betazero_b200.h; DESIGN.md section 2), derived from
the fourth frozen definition (endgame_ref.solve) rather than searched on its own: every legal move's value is replaced by
its sign (illegal actions stay -128), the root's value by the maximum of those signs (a finished game: the sign of its
disc difference), and the action by the first move in cell order whose sign is the root's -- the reference's strict ">"
on the signs, generally not the exact action.  A forced pass keeps 64 and a finished game 255; nodes are plain
negamax's count, an upper bound of any pruned search's.

    solve_wld(board, player)           the transform of endgame_ref.solve on the reference board API
    endgame_solve_wld(me, opp, size)   the transform of the C restatement (pyendgame.endgame_solve), batched in numpy
    wld_solver(solve)                  a selfplay_endgame_ref solver in WLD form: the WLD handover's restatement, whose
                                       solver_pi is uniform over the moves that keep the result and whose z is the
                                       exact handover's, since every move played keeps the handover position's result
"""
from __future__ import annotations

import numpy as np

from . import endgame_ref


def sign(x: int) -> int:
    return (x > 0) - (x < 0)


def to_wld(action: int, value: int, move_values):
    """one exact result (action, value, move_values[65]) in win/draw/loss form"""
    mv = [x if x == -128 else sign(x) for x in move_values]
    v = sign(value)
    if action < 64:
        action = mv.index(v)  # the pass's slot holds -128 when the mover has a move, so the first hit is a cell
    return action, v, mv


def solve_wld(board, player: int):
    """(action, value, move_values, nodes): endgame_ref.solve in win/draw/loss form"""
    a, v, mv, nodes = endgame_ref.solve(board, player)
    return (*to_wld(a, v, mv), nodes)


def to_wld_batch(action, value, move_value):
    """numpy form of to_wld over a batch: (action uint8 [n], value int8 [n], move_value int8 [n, 65])"""
    action, value, move_value = np.asarray(action), np.asarray(value), np.asarray(move_value)
    mv = np.where(move_value == -128, move_value, np.sign(move_value)).astype(np.int8)
    v = np.sign(value).astype(np.int8)
    first = np.argmax(mv[:, :64] == v[:, None], axis=1)  # the first move whose sign is the root's
    return np.where(action < 64, first, action).astype(np.uint8), v, mv


def endgame_solve_wld(me, opp, size: int = 8):
    """TEST INFRASTRUCTURE: the checker of bz_endgame_solve_wld -- the sign transform of pyendgame.endgame_solve (the C
    restatement without pruning): (action uint8 [n], value int8 [n], move_value int8 [n, 65], nodes int64 [n])"""
    from . import pyendgame

    act, val, mv, nodes = pyendgame.endgame_solve(me, opp, size)
    return (*to_wld_batch(act, val, mv), nodes)


def wld_solver(solve):
    """``solve(board, player) -> (action, value, move_values)`` (selfplay_endgame_ref.reference_solver / c_solver) in
    win/draw/loss form"""

    def solve_wld_(board, player):
        return to_wld(*solve(board, player))

    return solve_wld_
