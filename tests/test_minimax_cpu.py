"""CPU: the minimax definition (oracle/minimax_ref.py, run on the oracle's board class) against its C restatement without
pruning (oracle/minimax.c) -- move, root value and node count -- on random-playout positions of every stage of the game;
and against the reference's own OptimalPlayer when a checkout of the reference is present."""
import multiprocessing
import os
from concurrent.futures import ProcessPoolExecutor

import numpy as np
import pytest

# (size, max depth, positions): 8x8 to depth 4, 6x6 to depth 6, 4x4 to the deepest the kernel takes (8, the whole rest
# of the game from the positions with at most 8 empty cells)
SETS = [(8, 4, 1000), (6, 6, 400), (4, 8, 600)]
SEED = 9


def _positions(size, max_depth, n):
    from oracle import pyoracle as po

    me, opp = po.playout_boards(n, seed=100 + size, size=size)
    rng = np.random.default_rng(size)
    depth = rng.integers(0, max_depth + 1, n).astype(np.uint8)
    keys = rng.integers(0, 2**32, n).astype(np.uint64)
    return me, opp, depth, keys


def _definition(args):
    """(action, value, nodes, fell back to the random move, met a node without moves) of minimax_ref on oracle boards"""
    from oracle import minimax_ref as mr
    from oracle import pyoracle as po

    size, me, opp, depth, key = args
    b = po.OracleReversiBoard(size=size)
    b.board = po.wire_to_grid(me, opp, size, 1)
    m = mr.Minimax(1, depth, seed=SEED, game_key=key)
    a, v = m.search(b)
    fallback = a < 64 and (depth == 0 or v == -mr.INF)
    return a, v, m.nodes, fallback, m.stuck > (1 if a == mr.PASS else 0)


@pytest.fixture(scope="module")
def cases():
    out = []
    for size, dmax, n in SETS:
        me, opp, depth, keys = _positions(size, dmax, n)
        out += [(size, int(me[i]), int(opp[i]), int(depth[i]), int(keys[i])) for i in range(n)]
    # spawned workers: the parent may hold OpenMP and torch threads, which a fork would copy in a broken state
    with ProcessPoolExecutor(max_workers=os.cpu_count() or 1, mp_context=multiprocessing.get_context("spawn")) as ex:
        res = list(ex.map(_definition, out, chunksize=8))
    return out, res


def test_definition_equals_the_c_oracle(cases):
    from oracle import pyminimax as pm

    out, res = cases
    assert len(out) >= 2000
    for size, dmax, _ in SETS:
        idx = [i for i, c in enumerate(out) if c[0] == size]
        me = np.array([out[i][1] for i in idx], np.uint64)
        opp = np.array([out[i][2] for i in idx], np.uint64)
        depth = np.array([out[i][3] for i in idx], np.uint8)
        keys = np.array([out[i][4] for i in idx], np.uint64)
        a, v, nodes = pm.minimax_moves(me, opp, depth, keys, seed=SEED, size=size)
        for j, i in enumerate(idx):
            assert (int(a[j]), int(v[j]), int(nodes[j])) == res[i][:3], (size, out[i], res[i])
        assert set(depth.tolist()) == set(range(dmax + 1))


def test_the_set_meets_every_case(cases):
    """passes, finished games, the no-pass quirk inside the search and the random move (depth 0 and all-(-inf) roots)"""
    from oracle import minimax_ref as mr

    out, res = cases
    acts = [r[0] for r in res]
    assert mr.PASS in acts and mr.GAME_OVER in acts
    assert sum(r[4] for r in res) >= 20  # searches that met a node without moves in a game that was not over
    assert sum(r[3] for i, r in enumerate(res) if out[i][3] == 0) >= 100  # depth 0: RandomPlayer
    assert any(r[3] and out[i][3] > 0 for i, r in enumerate(res))  # every move worth -inf: the random move again


def test_philox_matches_the_kernel_constants():
    """the Python Philox is the one selfplay and the openings use: a known value of the self-play sampler"""
    from oracle import minimax_ref as mr

    # Philox4x32-10 with counter (0, 0, 0, 0) and key 0 (Random123's known-answer test, first word)
    assert mr.philox_u32(0, 0, 0) == 0x6627E8D5


def test_random_move_rule():
    from oracle import minimax_ref as mr

    for n in (1, 2, 7, 13):
        ks = [mr.random_move_index(3, g, 20, n) for g in range(200)]
        assert min(ks) >= 0 and max(ks) == n - 1


@pytest.mark.skipif(not __import__("oracle.ref_shim", fromlist=["available"]).available(),
                    reason="the reference checkout is not present (set BETAZERO_REFERENCE)")
def test_definition_equals_the_live_reference_optimal_player():
    """the reference's own OptimalPlayer on its own board class, wherever it does not fall back to random.choice"""
    from oracle import minimax_ref as mr
    from oracle import pyoracle as po
    from oracle import ref_shim

    RB = ref_shim.reversi_board_cls()
    Opt = ref_shim.reversi_players_mod().OptimalPlayer
    n_cmp = 0
    for size, dmax, n in [(8, 3, 150), (6, 4, 150), (4, 6, 150)]:
        me, opp, depth, keys = _positions(size, dmax, n)
        for i in range(n):
            grid = po.wire_to_grid(me[i], opp[i], size, 1)
            b = RB(size=size)
            b.board = grid.copy()
            if not b.generate_possible_moves(1) or depth[i] == 0:
                continue
            ours = mr.Minimax(1, int(depth[i]), seed=SEED, game_key=int(keys[i]))
            a, v = ours.search(b)
            if v == -mr.INF:
                continue  # the reference plays random.choice here
            ref = Opt(1, max_depth=int(depth[i]))
            r, c = ref.get_move(b)
            assert a == r * 8 + c, (size, i)
            n_cmp += 1
    assert n_cmp > 100
