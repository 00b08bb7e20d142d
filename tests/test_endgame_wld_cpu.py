"""CPU: the win/draw/loss result derived from the endgame definition (oracle/endgame_wld_ref.py solve_wld, on the oracle's
board class) against the sign transform of the C restatement (endgame_wld_ref.endgame_solve_wld) -- action, value, every
move value and nodes -- on late positions of 4x4, 6x6 and 8x8 games with 0 to 7 empty squares; the live reference's
board class when a checkout of the reference is present; the WLD handover's solver (endgame_wld_ref.wld_solver) with
selfplay_endgame_ref.solver_pi; and the argument checks of the WLD options."""
import multiprocessing
import os
from concurrent.futures import ProcessPoolExecutor

import numpy as np
import pytest

SETS = [(4, 200), (6, 250), (8, 250)]  # (size, positions)
MAX_EMPTIES = 7


def _late_positions(size, n, seed):
    """mover-relative positions with at most MAX_EMPTIES empties from random games: roots that must pass and finished
    games included"""
    from oracle import pyoracle as po

    rng = np.random.default_rng(seed)
    me, opp = [], []
    k = 0
    while len(me) < n:
        plies = size * size - 4 - int(rng.integers(0, MAX_EMPTIES + 1)) + int(rng.integers(0, 3))
        g, pl, _, _ = po.random_playout(size, seed * 100_003 + k, plies)
        k += 1
        m, o = po.grid_to_wire(g, pl)
        if size * size - bin(m | o).count("1") <= MAX_EMPTIES:
            me.append(m)
            opp.append(o)
    return np.array(me, np.uint64), np.array(opp, np.uint64)


def _definition(args):
    from oracle import endgame_wld_ref as ewr
    from oracle import pyoracle as po

    size, me, opp = args
    b = po.OracleReversiBoard(size=size)
    b.board = po.wire_to_grid(me, opp, size, 1)
    return ewr.solve_wld(b, 1)


@pytest.fixture(scope="module")
def cases():
    out = []
    for size, n in SETS:
        me, opp = _late_positions(size, n, seed=100 + size)
        out += [(size, int(me[i]), int(opp[i])) for i in range(n)]
    # spawned workers: the parent may hold OpenMP and torch threads, which a fork would copy in a broken state
    with ProcessPoolExecutor(max_workers=os.cpu_count() or 1, mp_context=multiprocessing.get_context("spawn")) as ex:
        res = list(ex.map(_definition, out, chunksize=8))
    return out, res


def test_solve_wld_equals_the_sign_transform_of_the_c_oracle(cases):
    from oracle import endgame_wld_ref as ewr
    from oracle import pyendgame as pe

    out, res = cases
    for size in {c[0] for c in out}:
        idx = [i for i, c in enumerate(out) if c[0] == size]
        me = np.array([out[i][1] for i in idx], np.uint64)
        opp = np.array([out[i][2] for i in idx], np.uint64)
        a, v, mv, nodes = ewr.endgame_solve_wld(me, opp, size)
        ea, ev, emv, _ = pe.endgame_solve(me, opp, size)
        for j, i in enumerate(idx):
            ra, rv, rmv, rn = res[i]
            assert (a[j], v[j], nodes[j]) == (ra, rv, rn), (size, i)
            assert mv[j].tolist() == rmv, (size, i)
        assert set(np.unique(mv).tolist()) <= {-128, -1, 0, 1} and set(np.unique(v).tolist()) <= {-1, 0, 1}
        assert np.array_equal(v, np.sign(ev)) and np.array_equal(mv != -128, emv != -128)
        played = a < 64
        assert (mv[played, a[played]] == v[played]).all()  # the action keeps the result ...
        for j in np.nonzero(played)[0]:
            assert (mv[j, :a[j]] != v[j]).all()  # ... and is the first move in cell order that does
        empties = size * size - np.array([bin(int(x)).count("1") for x in me | opp])
        assert set(empties.tolist()) == set(range(MAX_EMPTIES + 1)), size
    acts = np.array([r[0] for r in res])
    assert (acts == 64).any() and (acts == 255).any() and (acts < 64).any()
    vals = np.array([r[1] for r in res])
    assert (vals == 1).any() and (vals == 0).any() and (vals == -1).any()
    # the WLD action differs from the exact one where an earlier move keeps the result with a smaller margin
    assert any(ewr.to_wld(*exact[:3])[0] != exact[0] for exact in (_exact(c) for c in out[:200]))


def _exact(case):
    from oracle import endgame_ref as er
    from oracle import pyoracle as po

    size, me, opp = case
    b = po.OracleReversiBoard(size=size)
    b.board = po.wire_to_grid(me, opp, size, 1)
    return er.solve(b, 1)


def test_4x4_start_position_is_a_loss():
    from oracle import endgame_wld_ref as ewr

    me, opp = np.array([0x0000000000040200], np.uint64), np.array([0x0000000000020400], np.uint64)
    a, v, mv, _ = ewr.endgame_solve_wld(me, opp, 4)
    assert v[0] == -1 and a[0] == 2 and sorted(mv[0][mv[0] != -128].tolist()) == [-1, -1, -1, -1]


@pytest.mark.skipif(not __import__("oracle.ref_shim", fromlist=["available"]).available(),
                    reason="the reference checkout is not present (set BETAZERO_REFERENCE)")
def test_solve_wld_runs_on_the_live_reference_board():
    """the WLD result on the reference's own ReversiBoard equals the sign transform of the C oracle"""
    from oracle import endgame_wld_ref as ewr
    from oracle import pyoracle as po
    from oracle import ref_shim

    RB = ref_shim.reversi_board_cls()
    for size, n in [(8, 60), (6, 60), (4, 60)]:
        me, opp = _late_positions(size, n, seed=150 + size)
        a, v, mv, nodes = ewr.endgame_solve_wld(me, opp, size)
        for i in range(n):
            b = RB(size=size)
            b.board = po.wire_to_grid(me[i], opp[i], size, 1).copy()
            ra, rv, rmv, rn = ewr.solve_wld(b, 1)
            assert (a[i], v[i], nodes[i]) == (ra, rv, rn) and mv[i].tolist() == rmv, (size, i)


def test_wld_solver_and_solver_pi():
    """pi uniform over the moves that keep the result; the move the first of them; a pass and a finished game kept"""
    from oracle import endgame_wld_ref as ewr
    from oracle import selfplay_endgame_ref as ser

    mv = [-128] * 65
    mv[3], mv[10], mv[40], mv[63] = 4, -2, 6, 0
    solve = ewr.wld_solver(lambda board, player: (40, 6, list(mv)))
    a, v, wmv = solve(None, 1)
    assert (a, v) == (3, 1) and wmv[3] == wmv[40] == 1 and wmv[10] == -1 and wmv[63] == 0 and wmv[0] == -128
    pi = ser.solver_pi(wmv, v)
    assert pi.dtype == np.float32 and pi[3] == pi[40] == np.float32(0.5) and np.count_nonzero(pi) == 2
    assert ser.solver_pi(mv, 6)[40] == 1.0  # the exact pi: only the margin-maximising move
    mv = [-128] * 65
    mv[5], mv[9] = -3, 0
    a, v, wmv = ewr.wld_solver(lambda board, player: (9, 0, list(mv)))(None, 1)
    assert (a, v) == (9, 0) and ser.solver_pi(wmv, v)[9] == 1.0  # a draw kept: the loss is not a WLD-optimal move
    mv = [-128] * 65
    mv[64] = -6
    a, v, wmv = ewr.wld_solver(lambda board, player: (64, -6, list(mv)))(None, 1)
    assert (a, v) == (64, -1) and ser.solver_pi(wmv, v).tolist() == [0.0] * 64 + [1.0]  # a forced pass
    assert ewr.wld_solver(lambda board, player: (255, 3, [-128] * 65))(None, 1)[:2] == (255, 1)  # a finished game


@pytest.mark.parametrize("size,n_sims,empties", [(4, 24, 6), (6, 16, 8)])
def test_wld_restatement_keeps_the_prefix_and_z(size, n_sims, empties):
    """the WLD handover game: the records before the handover and the winner are those of the exact handover game; every
    solver record's pi covers the exact one's support"""
    from oracle import endgame_wld_ref as ewr
    from oracle import mcts_ref as mr
    from oracle import pyoracle as po
    from oracle import selfplay_endgame_ref as ser

    game = mr.ReversiGame(po.OracleReversiBoard, size)
    ev = lambda a, b: mr.hash_eval(a, b, 5, 65)  # noqa: E731
    he, we, pe_ = ser.self_play_game_endgame(game, n_sims, 1.25, ev, empties, solve=ser.c_solver(game))
    hw, ww, pw = ser.self_play_game_endgame(game, n_sims, 1.25, ev, empties, solve=ewr.wld_solver(ser.c_solver(game)))
    assert pe_ == pw and pw is not None and we == ww
    for x, y in zip(he[:pw], hw[:pw]):
        assert x[:3] == y[:3] and x[4] == y[4] and np.array_equal(x[3], y[3])
    assert ((he[pw][3] > 0) <= (hw[pw][3] > 0)).all()


def test_argument_checks_raise_before_touching_the_gpu():
    from betazero_b200 import loop, selfplay

    for bad in ("nope", "WLD", None, 1):
        with pytest.raises(ValueError, match="endgame_solve"):
            selfplay.BatchedSelfPlay(8, 8, None, endgame_empties=8, endgame_solve=bad)
    with pytest.raises(ValueError, match="endgame_solve"):
        selfplay.BatchedSelfPlay(8, 8, None, endgame_solve="nope")
    assert selfplay.check_endgame_solve("wld") == "wld" and selfplay.check_endgame_solve("exact") == "exact"
    assert loop.default_args().endgame_solve == "exact"
    with pytest.raises(ValueError, match="endgame_solve"):
        loop.LoopState(loop.default_args(endgame_solve="nope"), 0, 1)


def test_wld_metrics_report_wld_accuracy_only():
    from betazero_b200 import endgame

    L = -128
    mv = np.full((3, 65), L, np.int8)
    mv[0, [3, 5, 9]] = [4, 4, -2]
    mv[1, [0, 1]] = [-6, 0]
    mv[2, [10, 20, 30, 40]] = [-2, -10, 2, 1]
    value = np.array([4, 0, 2], np.int8)
    played = np.array([5, 0, 40])
    exact = endgame.move_metrics(mv, value, played)
    wmv, wv = np.where(mv == L, mv, np.sign(mv)).astype(np.int8), np.sign(value).astype(np.int8)
    w = endgame.move_metrics(wmv, wv, played, wld=True)
    assert w == {"wld_accuracy": exact["wld_accuracy"]}
    assert endgame.random_metrics(wmv, wv, wld=True) == {"wld_accuracy": endgame.random_metrics(mv, value)["wld_accuracy"]}
    assert endgame.value_metrics(np.array([0.5, -0.2, -0.1]), wv) == endgame.value_metrics(np.array([0.5, -0.2, -0.1]), value)
