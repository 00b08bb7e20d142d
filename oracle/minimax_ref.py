"""THE DEFINITION of the minimax players -- the reference's depth-limited ``OptimalPlayer`` and its ``RandomPlayer``
(src/reversi/players/reversi_players.py:26-77, as SURVEY.md section 3.2 records it), in the role oracle/mcts_ref.py has
for MCTS.  It calls only the reference board API (``generate_possible_moves``, ``make_move``, ``is_game_over``,
``get_score``, ``.board``), so it runs on the reference's own ``ReversiBoard`` and on ``pyoracle.OracleReversiBoard``.

    minimax(board, maximizing, depth)                                              reversi_players.py:46-69
        depth >= max_depth or board.is_game_over(): evaluate_board(board)          :47-48
        maximizing: over generate_possible_moves(symbol), row-major; keep a child only when strictly > the best  :50-59
        minimizing: over generate_possible_moves(-symbol); strictly <             :60-69
    evaluate_board: the disc difference from symbol's point of view (get_score)   :71-77, a plain count, no win bonus
    get_move: the search's move; none -> a random legal move                       :40-45

Kept quirk: there is no pass handling.  A node whose side has no move in a game that is not over returns the loop's
initial -inf (maximizing) or +inf (minimizing); the ABI writes them as -127 / +127.

Decided here where SURVEY.md is silent:
* The random move of get_move (:42-43, Python's ``random.choice``, not reproducible) is drawn as the openings draw
  theirs: ``u = philox_u32(seed, 2**32 + game_key, discs on the board)``, the k-th legal move in ascending cell order with
  ``k = floor(u * n_moves / 2**32)``.  The counter differs at every decision of one game, passes included; the key
  never meets an opening's (pair ids < 2**32).  ``RandomPlayer`` (:26-32) is ``max_depth = 0``: the search at depth 0
  returns the evaluation and no move, so every move is the random one.
* A root whose player has no move returns action 64 (a pass) and a finished game 255; the reference's get_move is never
  called there (reversi_terminal.py:22-32 passes without asking the player).
"""
from __future__ import annotations

import math

INF = 127  # the ABI's int8 for +-inf
PASS, GAME_OVER = 64, 255


def philox_u32(seed: int, key: int, counter: int) -> int:
    """Philox4x32-10: the first output word of counter block (key lo, key hi, counter, 0) under the 64-bit seed
    (betazero_b200/csrc/common.cuh philox_u32)."""
    M = 0xFFFFFFFF
    c0, c1, c2, c3 = key & M, (key >> 32) & M, counter & M, 0
    k0, k1 = seed & M, (seed >> 32) & M
    for _ in range(10):
        p0, p1 = 0xD2511F53 * c0, 0xCD9E8D57 * c2
        n0 = ((p1 >> 32) ^ c1 ^ k0) & M
        n2 = ((p0 >> 32) ^ c3 ^ k1) & M
        c1, c3, c0, c2 = p1 & M, p0 & M, n0, n2
        k0, k1 = (k0 + 0x9E3779B9) & M, (k1 + 0xBB67AE85) & M
    return c0


def random_move_index(seed: int, game_key: int, discs: int, n_moves: int) -> int:
    """index into the row-major move list of the random move"""
    u = philox_u32(seed, (1 << 32) + game_key, discs)
    return (u * n_moves) >> 32


def _clip(v) -> int:
    return INF if v == math.inf else (-INF if v == -math.inf else int(v))


class Minimax:
    """``OptimalPlayer(symbol, max_depth)`` of reversi_players.py:35-77 (``max_depth = 0``: ``RandomPlayer``)."""

    def __init__(self, symbol: int, max_depth: int, seed: int = 0, game_key: int = 0):
        self.symbol, self.max_depth, self.seed, self.game_key = int(symbol), int(max_depth), int(seed), int(game_key)
        self.nodes = 0
        self.stuck = 0  # nodes of the last search whose side had no move in a game that was not over (the quirk)

    def evaluate_board(self, board) -> int:
        _, (c1, c2) = board.get_score()  # counts of +1 (X) and -1 (O)
        return c1 - c2 if self.symbol == 1 else c2 - c1

    def minimax(self, board, maximizing: bool, depth: int):
        """(value, move): the reference's recursion, values as Python numbers with +-inf"""
        self.nodes += 1
        if depth >= self.max_depth or board.is_game_over():
            return self.evaluate_board(board), None
        if not board.generate_possible_moves(self.symbol if maximizing else -self.symbol):
            self.stuck += 1  # the loop below does not run
        if maximizing:
            best, best_move = -math.inf, None
            for r, c in board.generate_possible_moves(self.symbol):
                v, _ = self.minimax(board.make_move(r, c, self.symbol), False, depth + 1)
                if v > best:
                    best, best_move = v, (r, c)
            return best, best_move
        best, best_move = math.inf, None
        for r, c in board.generate_possible_moves(-self.symbol):
            v, _ = self.minimax(board.make_move(r, c, -self.symbol), True, depth + 1)
            if v < best:
                best, best_move = v, (r, c)
        return best, best_move

    def search(self, board):
        """(action, value): action = row*8 + col of the move get_move plays, 64 for a pass, 255 for a finished game;
        value = the root's minimax value with +-inf as +-127"""
        self.nodes = self.stuck = 0
        moves = board.generate_possible_moves(self.symbol)
        value, move = self.minimax(board, True, 0)
        if not moves:
            return (GAME_OVER if board.is_game_over() else PASS), _clip(value)
        if move is None:  # reversi_players.py:42-43
            discs = sum(1 for row in board.board for x in row if x != 0)
            move = moves[random_move_index(self.seed, self.game_key, discs, len(moves))]
        return move[0] * 8 + move[1], _clip(value)

    def get_move(self, board):
        a, _ = self.search(board)
        return (None, None) if a >= 64 else (a >> 3, a & 7)
