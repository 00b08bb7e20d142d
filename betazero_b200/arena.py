"""Arena / evaluation against reference-compatible players ("next" row 4 of SURVEY.md section 8f).

Plays any two objects with the reference's ``get_move(board) -> (row, col)`` interface on any
reference-compatible board class, in the order of ``ReversiTerminal.play``
(src/reversi/game_logic/reversi_terminal.py:16-38: moves?, get_move, make_move -- a ValueError
gives the same player another try --, pass when there is no move, is_game_over, flip player),
without the prints, and scores with ``get_score`` (reversi_board.py:67-76).

This path plays one game at a time and searches one tree per move.  To measure two nets against each other over
thousands of games use ``betazero_b200.match.BatchedMatch`` (every game of the match searched in the same launch, the
same moves as ``MCTSPlayer``s here).
"""
from __future__ import annotations


def play_game(board_cls, player1, player2, size: int = 8, max_retries: int = 3):
    """One game.  Returns (winner in {1, -1, 0}, (count_p1, count_p2), plies)."""
    board = board_cls(size=size)
    players = {1: player1, -1: player2}
    current, over, plies, retries = 1, False, 0, 0
    while not over:
        moves = board.generate_possible_moves(current)
        if moves:
            row, col = players[current].get_move(board)
            try:
                board = board.make_move(row, col, current)
            except ValueError:
                retries += 1
                if retries > max_retries:
                    raise
                continue  # reversi_terminal.py:28-30: same player retries
            retries = 0
        over = board.is_game_over()
        current *= -1
        plies += 1
    winner, counts = board.get_score()
    return winner, counts, plies


def play_match(board_cls, make_p1, make_p2, n_games: int = 10, size: int = 8) -> dict:
    """n_games with colours alternating; ``make_pX(symbol)`` builds a player for that colour.
    Returns wins/draws/losses from the point of view of the first factory."""
    res = {"wins": 0, "draws": 0, "losses": 0, "disc_diff": 0}
    for g in range(n_games):
        first_is_x = g % 2 == 0
        px, po = (make_p1(1), make_p2(-1)) if first_is_x else (make_p2(1), make_p1(-1))
        winner, (c1, c2), _ = play_game(board_cls, px, po, size)
        mine = 1 if first_is_x else -1
        res["wins" if winner == mine else "draws" if winner == 0 else "losses"] += 1
        res["disc_diff"] += (c1 - c2) * mine
    return res
