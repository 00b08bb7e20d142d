"""CPU tests: pin the C oracle (oracle/oracle.c) against outputs of the reference itself.

tests/golden/reversi_env.npz and ttt_env.npz were produced by oracle/make_golden.py running the
LIVE reference (reversi_board.py / tic_tac_toe_board.py); ttt_env.npz also carries the
reference's only golden file, tic_tac_toe_data.csv.  The oracle is checked against them through its batched
wire-format functions and through its board classes.
"""
import numpy as np
import pytest

from oracle import pyoracle as po


@pytest.mark.parametrize("size", [4, 6, 8])
def test_oracle_matches_reference_outputs(golden_env, size):
    g = golden_env
    me, opp = g[f"s{size}_me"], g[f"s{size}_opp"]
    assert np.array_equal(po.legal_mask(me, opp, size), g[f"s{size}_mask"])
    assert np.array_equal(po.legal_mask(opp, me, size), g[f"s{size}_mask_opp"])
    over, win, cm, co = po.terminal(me, opp, size)
    assert np.array_equal(over, g[f"s{size}_over"])
    assert np.array_equal(win, g[f"s{size}_winner"])
    assert np.array_equal(cm, g[f"s{size}_cnt_me"]) and np.array_equal(co, g[f"s{size}_cnt_opp"])
    idx, act = g[f"s{size}_succ_idx"], g[f"s{size}_succ_act"]
    mo, oo, err = po.apply(me[idx], opp[idx], act, size)
    assert not err.any()
    assert np.array_equal(mo, g[f"s{size}_succ_me"]) and np.array_equal(oo, g[f"s{size}_succ_opp"])
    bidx, bact = g[f"s{size}_bad_idx"], g[f"s{size}_bad_act"]
    _, _, err = po.apply(me[bidx], opp[bidx], bact, size)
    assert err.all()  # the reference raised ValueError("Invalid move") on each of these


def test_oracle_board_class_replays_reference_demo(golden_env):
    # reversi_board.py:92-99 demo on 4x4; expected boards recorded from the reference
    b = po.OracleReversiBoard(size=4)
    demo = golden_env["demo4_boards"]
    assert np.array_equal(b.board, demo[0])
    for k, (r, c, p) in enumerate(((0, 2, 1), (0, 1, -1), (2, 0, 1))):
        b = b.make_move(r, c, p)
        assert np.array_equal(b.board, demo[k + 1])
    assert b.is_valid_move(0, 3, -1) == bool(golden_env["demo4_valid_0_3_m1"])
    with pytest.raises(ValueError, match="Invalid move"):
        b.make_move(0, 2, 1)  # occupied cell


@pytest.mark.parametrize("size", [4, 6, 8])
def test_oracle_episode_matches_reference(golden_env, size):
    # full reference episode (reversi_terminal.py:16-38 order): replay its actions through the oracle
    g = golden_env
    me, opp, act = g[f"ep{size}_me"], g[f"ep{size}_opp"], g[f"ep{size}_action"]
    for k in range(len(act) - 1):
        m, o, err = po.apply(me[k:k + 1], opp[k:k + 1], act[k:k + 1], size)
        assert err[0] == 0 and m[0] == me[k + 1] and o[0] == opp[k + 1]
    m, o, err = po.apply(me[-1:], opp[-1:], act[-1:], size)
    over, win, cm, co = po.terminal(m, o, size)
    assert over[0] == 1
    final = g[f"ep{size}_final"]
    w, c1, c2 = g[f"ep{size}_score"]
    b = po.OracleReversiBoard(size=size)
    b.board = final.astype(np.int64)
    assert b.is_game_over() and b.get_score() == (w, (c1, c2))


def test_ttt_oracle_matches_reference_outputs(golden_ttt):
    g = golden_ttt
    assert np.array_equal(po.ttt_legal_mask(g["x"], g["o"]), g["mask"])
    over, win = po.ttt_terminal(g["x"], g["o"])
    assert np.array_equal(over, g["over"]) and np.array_equal(win, g["winner"])


def test_ttt_csv_golden(golden_ttt):
    """tic_tac_toe_data.csv: canonical states (mover = +1) and one-hot actions of optimal play.
    Pins canonical form (generate_training_games.py:17-21) and move application."""
    st, ac = golden_ttt["csv_state"], golden_ttt["csv_action"]
    assert st.shape == (180, 9) and ac.shape == (180, 9)
    for s, a in zip(st, ac):
        assert a.sum() == 1 and set(np.unique(a)) <= {0, 1}
        k = int(np.argmax(a))
        # canonical: the mover is +1, so it has as many marks as the opponent, or one fewer
        assert (s == -1).sum() - (s == 1).sum() in (0, 1)
        b = po.OracleTicTacToeBoard(s.reshape(3, 3).astype(np.int64))
        assert b.is_game_over() == (False, None)
        assert (k // 3, k % 3) in b.generate_possible_moves()
        nb = b.make_move(k // 3, k % 3, 1)
        assert nb.board[k // 3, k % 3] == 1
        # wire-format equivalents
        x = sum(1 << i for i in range(9) if s[i] == 1)
        o = sum(1 << i for i in range(9) if s[i] == -1)
        xo, oo, err = po.ttt_apply([x], [o], [k], [1])
        assert err[0] == 0 and xo[0] == x | (1 << k) and oo[0] == o
    # consecutive rows of one game: next state == -(state + action) (generate_training_games.py:21)
    follows = sum(np.array_equal(st[i + 1], -(st[i] + ac[i])) for i in range(179))
    assert follows >= 180 - 20 - 20  # 20 games: every in-game transition must follow the rule


def _bits(mask):
    return [k for k in range(64) if (int(mask) >> k) & 1]


def test_oracle_vs_live_reference_random_boards(golden_env):
    """The board class (generate_possible_moves, make_move, is_game_over, get_score) against the answers of the
    reference's ReversiBoard recorded in reversi_env.npz, on a seeded sample of 150 boards per size; the order of
    generate_possible_moves against the move the reference episodes picked from its list (moves[len(moves) // 2])."""
    g = golden_env
    rng = np.random.default_rng(123)
    for size in (4, 6, 8):
        me, opp = g[f"s{size}_me"], g[f"s{size}_opp"]
        succ_idx, bad_idx = g[f"s{size}_succ_idx"], g[f"s{size}_bad_idx"]
        for i in np.sort(rng.choice(len(me), 150, replace=False)):
            ob = po.OracleReversiBoard(size=size)
            ob.board = po.wire_to_grid(me[i], opp[i], size)
            for p, key in ((1, "mask"), (-1, "mask_opp")):
                assert [r * 8 + c for r, c in ob.generate_possible_moves(p)] == _bits(g[f"s{size}_{key}"][i])
            for j in np.flatnonzero(succ_idx == i):
                a = int(g[f"s{size}_succ_act"][j])
                nb = ob.make_move(a >> 3, a & 7, 1)
                assert po.grid_to_wire(nb.board, -1) == (int(g[f"s{size}_succ_me"][j]), int(g[f"s{size}_succ_opp"][j]))
            for j in np.flatnonzero(bad_idx == i):
                a = int(g[f"s{size}_bad_act"][j])
                with pytest.raises(ValueError, match="Invalid move"):
                    ob.make_move(a >> 3, a & 7, 1)
            assert ob.is_game_over() == bool(g[f"s{size}_over"][i])
            assert ob.get_score() == (int(g[f"s{size}_winner"][i]), (int(g[f"s{size}_cnt_me"][i]), int(g[f"s{size}_cnt_opp"][i])))
        for m, o, a in zip(g[f"ep{size}_me"], g[f"ep{size}_opp"], g[f"ep{size}_action"]):
            ob = po.OracleReversiBoard(size=size)
            ob.board = po.wire_to_grid(m, o, size)
            moves = ob.generate_possible_moves(1)
            assert (moves[len(moves) // 2] if moves else None) == (None if a == 64 else (a >> 3, a & 7))


def test_ttt_oracle_vs_live_reference(golden_ttt):
    """The board class (is_game_over, generate_possible_moves) against the answers of the reference's TicTacToeBoard
    recorded in ttt_env.npz, on all 3^9 grids."""
    g = golden_ttt
    for x, o, mask, over, winner in zip(g["x"], g["o"], g["mask"], g["over"], g["winner"]):
        grid = np.array([1 if (x >> k) & 1 else -1 if (o >> k) & 1 else 0 for k in range(9)], np.int64).reshape(3, 3)
        ob = po.OracleTicTacToeBoard(grid)
        assert ob.is_game_over() == (bool(over), None if winner == 2 else int(winner))
        assert [r * 3 + c for r, c in ob.generate_possible_moves()] == _bits(mask)


def test_board_generators_are_seeded():
    a = po.synthetic_boards(1000, seed=0)
    b = po.synthetic_boards(1000, seed=0)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    assert not (a[0] & a[1]).any()
    m, o = po.playout_boards(64, seed=0)
    assert not (m & o).any()
    # reachable boards keep the four centre cells occupied
    centre = np.uint64((1 << 27) | (1 << 28) | (1 << 35) | (1 << 36))
    assert (((m | o) & centre) == centre).all()
