"""THE DEFINITION of the exact endgame value -- the perfect player of bz_endgame_solve (include/betazero_b200.h;
DESIGN.md section 2), in the role oracle/minimax_ref.py has for the depth-limited minimax.  It calls only the reference
board API (``generate_possible_moves``, ``make_move``, ``is_game_over``, ``get_score``), so it runs on the reference's own
``ReversiBoard`` and on ``pyoracle.OracleReversiBoard``.

    value(board, player): player has moves -> max over them of -value(child, -player)
                          else the opponent has moves (a pass, reversi_terminal.py:31-35) -> -value(board, -player)
                          else (game over) player's discs - the opponent's (get_score, reversi_board.py:67-85):
                          empty squares go to nobody

Plain negamax, no pruning: every position entered counts one node, the positions after passes included.
"""
from __future__ import annotations

PASS, GAME_OVER = 64, 255


def _negamax(board, player: int, nodes: list) -> int:
    nodes[0] += 1
    moves = board.generate_possible_moves(player)
    if moves:
        return max(-_negamax(board.make_move(r, c, player), -player, nodes) for r, c in moves)
    if not board.is_game_over():
        return -_negamax(board, -player, nodes)
    _, (c1, c2) = board.get_score()
    return c1 - c2 if player == 1 else c2 - c1


def solve(board, player: int):
    """(action, value, move_values, nodes) of the position with ``player`` to move: action = row*8 + col of the first
    best move in cell order (the reference's strict ">"), 64 for a forced pass, 255 for a finished game; value = the
    exact final disc difference for ``player``; move_values: 65 ints, -value(child) of every legal move, the pass's at
    index 64, -128 elsewhere; nodes: positions entered, the root included."""
    player = int(player)
    nodes = [1]
    mv = [-128] * 65
    moves = board.generate_possible_moves(player)
    if moves:
        for r, c in moves:
            mv[r * 8 + c] = -_negamax(board.make_move(r, c, player), -player, nodes)
        value = max(mv[:64])
        return mv.index(value), value, mv, nodes[0]
    if not board.is_game_over():
        mv[64] = -_negamax(board, -player, nodes)
        return PASS, mv[64], mv, nodes[0]
    _, (c1, c2) = board.get_score()
    return GAME_OVER, (c1 - c2 if player == 1 else c2 - c1), mv, nodes[0]
