"""Shared test helpers: the reference's episode loops restated without prints, and an oracle-side
MCTS player (oracle/mcts_ref.py on the C-restated boards) with the reference's player interface."""
import ctypes

import numpy as np
import pytest

from oracle import mcts_ref as mr
from oracle import pyoracle as po


def play_reversi_episode(board_cls, player1, player2, size=8, max_iters=200):
    """ReversiTerminal.play (src/reversi/game_logic/reversi_terminal.py:16-38) minus the prints.
    Returns (final board, list of (player, move or None))."""
    board = board_cls(size=size)
    players = {1: player1, -1: player2}
    current_player, game_over, trace = 1, False, []
    while not game_over and len(trace) < max_iters:
        moves = board.generate_possible_moves(current_player)
        if moves:
            row, col = players[current_player].get_move(board)
            board = board.make_move(row, col, current_player)
            trace.append((current_player, (row, col)))
        else:
            trace.append((current_player, None))
        game_over = board.is_game_over()
        current_player *= -1
    return board, trace


def play_ttt_headless(board_cls, player1, player2):
    """TicTacToeHeadless.play (src/tic_tac_toe/tic_tac_toe.py:13-34): returns (positions, winner)."""
    board = board_cls()
    players = {1: player1, -1: player2}
    current_player, game_over, winner, positions = 1, False, None, []
    while not game_over:
        positions.append(board.board)
        row, col = players[current_player].get_move(board)
        board = board.make_move(row, col, current_player)
        game_over, winner = board.is_game_over()
        current_player *= -1
        if game_over:
            positions.append(board.board)
    return positions, winner


class OracleMCTSPlayer:
    """get_move(board) -> (row, col) from the sequential Python MCTS definition + hash evaluator."""

    def __init__(self, symbol, n_sims, game="reversi", size=8, c_puct=1.25, salt=0):
        self.symbol, self.n_sims, self.c_puct, self.salt = symbol, n_sims, c_puct, salt
        self.is_ttt = game == "ttt"
        self.game = mr.TicTacToeGame(po.OracleTicTacToeBoard) if self.is_ttt else mr.ReversiGame(po.OracleReversiBoard, size)
        self.last_counts = None

    def get_move(self, board):
        A = self.game.n_actions
        m = mr.MCTS(self.game, self.c_puct, lambda a, b: mr.hash_eval(a, b, self.salt, A))
        # rebuild an oracle board from the caller's grid so any board class can be passed in
        if self.is_ttt:
            ob = po.OracleTicTacToeBoard(np.asarray(board.board))
        else:
            ob = po.OracleReversiBoard(size=board.size)
            ob.board = np.asarray(board.board).copy()
        m.reset(ob, self.symbol)
        m.run(self.n_sims)
        cnt, _, _ = m.root_stats()
        self.last_counts = cnt
        a = mr.pick_move(cnt)
        if cnt.sum() == 0 or (not self.is_ttt and a == 64):
            return None, None
        return (a // 3, a % 3) if self.is_ttt else (a >> 3, a & 7)


@pytest.fixture(scope="module", autouse=True)
def _minimax_bounds_checks():
    """a -DBZ_BOUNDS_CHECK library: the violation record of the minimax and solver kernels (minimax.cu has its own) must
    stay empty.  Imported by the test modules of those kernels."""
    yield
    import torch

    from betazero_b200 import _lib

    if _lib._lib is not None and hasattr(_lib._lib, "bz_debug_checks_minimax"):
        torch.cuda.synchronize()
        rec = (ctypes.c_int * 4)()
        assert _lib._lib.bz_debug_checks_minimax(rec) == 0
        assert rec[3] == 0, f"check {rec[0]} failed in block {rec[1]}, thread {rec[2]} ({rec[3]} violations)"
