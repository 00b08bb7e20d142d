"""The alpha-beta searches' node counts, pinned: bz_minimax_moves, the minimax entrants of a tournament,
bz_endgame_solve and bz_endgame_solve_wld against golden/alphabeta_nodes.npz, bit for bit in action, value, move values
and nodes per root.  The other tests bound node counts only (at most plain minimax / negamax), so a change of move order
or of a cutoff would pass them; node counts are what sets the solvers' speed.

The golden was written on a B200 by the library before the two searches became one:
    python tests/test_gpu_alphabeta_nodes.py --write
The inputs come from the seeds below, so the writer and the test run the same code."""
import os
import sys

import numpy as np
import pytest

TESTS = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(TESTS)
for p in (ROOT, TESTS):  # run as a script (--write): the repository and the helpers
    if p not in sys.path:
        sys.path.insert(0, p)

from helpers import _minimax_bounds_checks  # noqa: E402,F401

GOLDEN = os.path.join(TESTS, "golden", "alphabeta_nodes.npz")

pytestmark = pytest.mark.gpu

# (name, size, roots, depths): random-playout roots of every stage (passes and finished games included), depths drawn
# uniformly from the list
MINIMAX_SETS = [
    ("mm8", 8, 640, [1, 2, 3, 4, 5]),
    ("mm8d6", 8, 96, [6]),
    ("mm6", 6, 384, list(range(0, 8))),
    ("mm4", 4, 256, list(range(0, 9))),
]
# (name, size, roots, empties): endgame.positions suites (8x8), or late random-playout positions with 0 .. empties
# empty squares (6x6, 4x4: passes and finished games included)
SOLVE_SETS = [
    ("eg8e8", 8, 256, 8),
    ("eg8e10", 8, 256, 10),
    ("eg8e12", 8, 128, 12),
    ("eg6", 6, 192, 12),
    ("eg4", 4, 128, 12),
]
WLD_ONLY_SETS = [("eg8e14", 8, 64, 14)]
TOURNAMENT = dict(depths=(2, 3), games_per_pairing=8, board_size=6, seed=11)


def _dev(x):
    from betazero_b200 import env

    return env.to_device_u64(np.ascontiguousarray(x, np.uint64))


def _minimax_roots(size, n, depths, seed):
    from oracle import pyoracle as po

    me, opp = po.playout_boards(n, seed=seed, size=size)
    rng = np.random.default_rng(seed)
    depth = rng.choice(np.array(depths, np.uint8), n)
    return me, opp, depth, rng.integers(0, 2**32, n).astype(np.uint64)


def _late_positions(size, n, max_empties, seed):
    from oracle import pyoracle as po

    rng = np.random.default_rng(seed)
    me, opp = [], []
    k = 0
    while len(me) < n:
        plies = size * size - 4 - int(rng.integers(0, max_empties + 1))
        g, pl, _, _ = po.random_playout(size, seed * 100_003 + k, plies)
        k += 1
        m, o = po.grid_to_wire(g, pl)
        if size * size - bin(m | o).count("1") <= max_empties:
            me.append(m)
            opp.append(o)
    return np.array(me, np.uint64), np.array(opp, np.uint64)


def _solve_roots(size, n, empties, seed):
    from betazero_b200 import endgame, env

    if size == 8:
        s = endgame.positions(n, empties, 8, seed=seed)
        return env.to_host_u64(s.me), env.to_host_u64(s.opp)
    return _late_positions(size, n, empties, seed)


def compute():
    """every pinned array, keyed by set and field; the inputs are stored too, so a change of the generators shows"""
    import torch

    from betazero_b200 import minimax, tournament

    out = {}
    for i, (name, size, n, depths) in enumerate(MINIMAX_SETS):
        me, opp, depth, keys = _minimax_roots(size, n, depths, seed=100 + i)
        a, v, nodes = minimax.best_moves(_dev(me), _dev(opp), torch.from_numpy(depth.astype(np.int64)), size=size,
                                         seed=29, keys=torch.from_numpy(keys.astype(np.int64)))
        out.update({f"{name}/me": me, f"{name}/opp": opp, f"{name}/depth": depth, f"{name}/action": a.cpu().numpy(),
                    f"{name}/value": v.cpu().numpy(), f"{name}/nodes": nodes.cpu().numpy()})
    for wld, sets in ((False, SOLVE_SETS), (True, SOLVE_SETS + WLD_ONLY_SETS)):
        for i, (name, size, n, empties) in enumerate(sets):
            me, opp = _solve_roots(size, n, empties, seed=200 + i)
            a, v, mv, nodes = minimax.solve(_dev(me), _dev(opp), size, wld=wld)
            key = f"{name}{'w' if wld else ''}"
            out.update({f"{key}/me": me, f"{key}/opp": opp, f"{key}/action": a.cpu().numpy(),
                        f"{key}/value": v.cpu().numpy(), f"{key}/move_value": mv.cpu().numpy(),
                        f"{key}/nodes": nodes.cpu().numpy()})
    T = TOURNAMENT
    t = tournament.Tournament([tournament.Minimax(d) for d in T["depths"]], T["games_per_pairing"],
                              board_size=T["board_size"], seed=T["seed"])
    r = t.play()
    out["tournament/moves"] = np.asarray(r["moves"])
    out["tournament/minimax_nodes"] = np.array([r["minimax_nodes"]], np.int64)
    return out


@pytest.fixture(scope="module")
def pinned():
    return compute(), np.load(GOLDEN)


def _fields(prefix, g):
    return sorted(k for k in g.files if k.startswith(prefix + "/"))


@pytest.mark.parametrize("name", [s[0] for s in MINIMAX_SETS])
def test_minimax_moves_and_nodes(pinned, name):
    got, g = pinned
    fields = _fields(name, g)
    assert {f.split("/")[1] for f in fields} == {"me", "opp", "depth", "action", "value", "nodes"}
    for f in fields:
        assert np.array_equal(got[f], g[f]), f


@pytest.mark.parametrize("name", [s[0] for s in SOLVE_SETS] + [s[0] + "w" for s in SOLVE_SETS + WLD_ONLY_SETS])
def test_solver_moves_and_nodes(pinned, name):
    got, g = pinned
    fields = _fields(name, g)
    assert {f.split("/")[1] for f in fields} == {"me", "opp", "action", "value", "move_value", "nodes"}
    for f in fields:
        assert np.array_equal(got[f], g[f]), f


def test_minimax_tournament_moves_and_nodes(pinned):
    got, g = pinned
    assert int(g["tournament/minimax_nodes"][0]) > 0
    for f in ("tournament/moves", "tournament/minimax_nodes"):
        assert np.array_equal(got[f], g[f]), f


def test_every_root_kind_is_pinned(pinned):
    """the sets hold roots that must pass, finished games and every depth / empties they name"""
    _, g = pinned
    for name, size, n, depths in MINIMAX_SETS:
        assert set(g[f"{name}/depth"].tolist()) == set(depths) and len(g[f"{name}/nodes"]) == n
    for name in ("mm6", "mm4", "eg6", "eg4", "eg6w", "eg4w"):
        assert (g[f"{name}/action"] == 64).any() and (g[f"{name}/action"] == 255).any(), name


if __name__ == "__main__":
    if sys.argv[1:] != ["--write"]:
        sys.exit("usage: python tests/test_gpu_alphabeta_nodes.py --write")
    arrays = compute()
    np.savez_compressed(GOLDEN, **arrays)
    print(GOLDEN, os.path.getsize(GOLDEN), "bytes")
