"""CPU: the endgame solver's definition (oracle/endgame_ref.py solve, run on the oracle's board class) against its C
restatement (oracle/endgame.c orc_endgame_solve) -- action, value, every move value and nodes -- on late positions of
4x4, 6x6 and 8x8 games with 0 to 7 empty squares; the 4x4 start position's value; the live reference's board class when
a checkout of the reference is present; and the metric arithmetic of betazero_b200/endgame.py."""
import multiprocessing
import os
from concurrent.futures import ProcessPoolExecutor

import numpy as np
import pytest

SETS = [(4, 300), (6, 350), (8, 350)]  # (size, positions)
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
    from oracle import endgame_ref as er
    from oracle import pyoracle as po

    size, me, opp = args
    b = po.OracleReversiBoard(size=size)
    b.board = po.wire_to_grid(me, opp, size, 1)
    return er.solve(b, 1)


@pytest.fixture(scope="module")
def cases():
    out = []
    for size, n in SETS:
        me, opp = _late_positions(size, n, seed=size)
        out += [(size, int(me[i]), int(opp[i])) for i in range(n)]
    # spawned workers: the parent may hold OpenMP and torch threads, which a fork would copy in a broken state
    with ProcessPoolExecutor(max_workers=os.cpu_count() or 1, mp_context=multiprocessing.get_context("spawn")) as ex:
        res = list(ex.map(_definition, out, chunksize=8))
    return out, res


def test_definition_equals_the_c_oracle(cases):
    from oracle import pyendgame as pe

    out, res = cases
    for size in {c[0] for c in out}:
        idx = [i for i, c in enumerate(out) if c[0] == size]
        me = np.array([out[i][1] for i in idx], np.uint64)
        opp = np.array([out[i][2] for i in idx], np.uint64)
        a, v, mv, nodes = pe.endgame_solve(me, opp, size)
        for j, i in enumerate(idx):
            ra, rv, rmv, rn = res[i]
            assert (a[j], v[j], nodes[j]) == (ra, rv, rn), (size, i)
            assert mv[j].tolist() == rmv, (size, i)
        empties = size * size - np.array([bin(int(x)).count("1") for x in me | opp])
        assert set(empties.tolist()) == set(range(MAX_EMPTIES + 1)), size
    acts = np.array([r[0] for r in res])
    assert (acts == 64).any() and (acts == 255).any() and (acts < 64).any()
    # passes inside the tree: roots with a move after which the opponent must pass
    from oracle import pyoracle as po

    def child_passes(size, me, opp):
        b = po.OracleReversiBoard(size=size)
        b.board = po.wire_to_grid(me, opp, size, 1)
        for r, c in b.generate_possible_moves(1):
            ch = b.make_move(r, c, 1)
            if not ch.generate_possible_moves(-1) and not ch.is_game_over():
                return True
        return False

    assert sum(child_passes(*c) for c in out) >= 10


def test_4x4_start_position_is_worth_minus_8():
    """the published 4x4 result: White wins 11-3, so the first player's value is -8"""
    from oracle import pyendgame as pe

    me, opp = np.array([0x0000000000040200], np.uint64), np.array([0x0000000000020400], np.uint64)
    a, v, mv, nodes = pe.endgame_solve(me, opp, 4)
    assert v[0] == -8 and a[0] == 2 and sorted(mv[0][mv[0] != -128].tolist()) == [-8, -8, -8, -8]
    assert 200_000 < nodes[0] < 250_000


@pytest.mark.skipif(not __import__("oracle.ref_shim", fromlist=["available"]).available(),
                    reason="the reference checkout is not present (set BETAZERO_REFERENCE)")
def test_definition_runs_on_the_live_reference_board():
    """the definition on the reference's own ReversiBoard equals the C oracle"""
    from oracle import endgame_ref as er
    from oracle import pyendgame as pe
    from oracle import pyoracle as po
    from oracle import ref_shim

    RB = ref_shim.reversi_board_cls()
    for size, n in [(8, 60), (6, 60), (4, 60)]:
        me, opp = _late_positions(size, n, seed=50 + size)
        a, v, mv, nodes = pe.endgame_solve(me, opp, size)
        for i in range(n):
            b = RB(size=size)
            b.board = po.wire_to_grid(me[i], opp[i], size, 1).copy()
            ra, rv, rmv, rn = er.solve(b, 1)
            assert (a[i], v[i], nodes[i]) == (ra, rv, rn) and mv[i].tolist() == rmv, (size, i)


def test_metric_arithmetic():
    from betazero_b200 import endgame

    L = -128
    mv = np.full((3, 65), L, np.int8)
    mv[0, [3, 5, 9]] = [4, 4, -2]     # best 4, two optimal moves of three
    mv[1, [0, 1]] = [-6, 0]           # best 0 (a draw), one optimal of two
    mv[2, [10, 20, 30, 40]] = [-2, -10, 2, 1]  # best 2
    value = np.array([4, 0, 2], np.int8)
    r = endgame.move_metrics(mv, value, np.array([5, 0, 40]))
    assert r["move_accuracy"] == pytest.approx(1 / 3)
    assert r["wld_accuracy"] == pytest.approx(2 / 3)  # +4 / +4, -6 / 0 lost the draw, +1 / +2 keeps the win
    assert r["mean_disc_loss"] == pytest.approx((0 + 6 + 1) / 3)
    rnd = endgame.random_metrics(mv, value)
    assert rnd["move_accuracy"] == pytest.approx((2 / 3 + 1 / 2 + 1 / 4) / 3)
    assert rnd["wld_accuracy"] == pytest.approx((2 / 3 + 1 / 2 + 2 / 4) / 3)
    assert rnd["mean_disc_loss"] == pytest.approx(((0 + 0 + 6) / 3 + (6 + 0) / 2 + (4 + 12 + 0 + 1) / 4) / 3)
    vm = endgame.value_metrics(np.array([0.5, -0.2, -0.1]), value)
    assert vm["value_sign_accuracy"] == pytest.approx(1 / 2)  # the draw is not decided
    assert vm["value_mse"] == pytest.approx(((0.5 - 1) ** 2 + 0.2 ** 2 + 1.1 ** 2) / 3)
    with pytest.raises(ValueError):
        endgame.move_metrics(mv, value, np.array([4, 0, 40]))  # cell 4 is not legal in position 0
