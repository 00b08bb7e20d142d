"""CPU: the sequential restatement of self-play with the endgame handover (oracle/selfplay_endgame_ref.py), the layout of
bz_selfplay_endgame_state against the C compiler, and the argument checks of the handover options."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import mcts_ref as mr
from oracle import pyoracle as po
from oracle import selfplay_endgame_ref as ser

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "betazero_b200.h")


def _game(size, n_sims, salt, empties, solve=None, leaves=1):
    game = mr.ReversiGame(po.OracleReversiBoard, size)
    ev = lambda a, b: mr.hash_eval(a, b, salt, 65)  # noqa: E731
    out = ser.self_play_game_endgame(game, n_sims, 1.25, ev, empties, solve=solve or ser.c_solver(game), leaves=leaves)
    return game, ev, out


def test_endgame_state_layout_matches_the_c_compiler(tmp_path):
    from betazero_b200._lib import BzSelfplayEndgameState

    fields = [n for n, _ in BzSelfplayEndgameState._fields_]
    prog = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', "int main(void){",
            'printf("%zu\\n", sizeof(bz_selfplay_endgame_state));']
    prog += [f'printf("%zu\\n", offsetof(bz_selfplay_endgame_state, {f}));' for f in fields]
    prog += ["return 0;}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(prog))
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-o", str(exe), str(src)])
    vals = [int(v) for v in subprocess.check_output([str(exe)], text=True).split()]
    assert vals == [C.sizeof(BzSelfplayEndgameState)] + [getattr(BzSelfplayEndgameState, f).offset for f in fields]
    assert fields[:BzSelfplayEndgameState.N_SCALARS] == ["empties", "cap", "max_plies", "reserved"]


def test_solver_pi_is_uniform_over_the_optimal_moves():
    mv = [-128] * 65
    mv[3], mv[10], mv[40], mv[63] = 4, -2, 4, 4
    pi = ser.solver_pi(mv, 4)
    assert pi.dtype == np.float32 and pi[3] == pi[40] == pi[63] == np.float32(1) / np.float32(3)
    assert np.count_nonzero(pi) == 3
    mv = [-128] * 65
    mv[64] = -6
    assert ser.solver_pi(mv, -6).tolist() == [0.0] * 64 + [1.0]  # a forced pass


@pytest.mark.parametrize("size,n_sims,empties", [(4, 24, 6), (4, 16, 11), (6, 16, 8)])
def test_the_reference_and_the_c_solver_play_the_same_game(size, n_sims, empties):
    game = mr.ReversiGame(po.OracleReversiBoard, size)
    _, _, a = _game(size, n_sims, 3, empties, solve=ser.reference_solver)
    _, _, b = _game(size, n_sims, 3, empties, solve=ser.c_solver(game))
    (ha, wa, pa), (hb, wb, pb) = a, b
    assert pa == pb and pa is not None and wa == wb and len(ha) == len(hb)
    for x, y in zip(ha, hb):
        assert x[:3] == y[:3] and x[4] == y[4] and np.array_equal(x[3], y[3])


@pytest.mark.parametrize("size,n_sims,empties,leaves", [(4, 24, 6, 1), (6, 16, 10, 1), (6, 16, 10, 2), (8, 32, 8, 1)])
def test_restatement_prefix_moves_and_outcome(size, n_sims, empties, leaves):
    """the records up to the handover are self_play_game's; every later record is a perfect move with pi uniform over
    the optimal moves; the winner is the sign of the handover position's exact value"""
    from oracle import pyendgame as pe

    game, ev, (hist, winner, h) = _game(size, n_sims, 5, empties, leaves=leaves)
    full, _ = mr.self_play_game(game, n_sims, 1.25, ev, leaves=leaves)
    assert h is not None and 0 < h < len(hist)
    for k in range(h):
        me, opp, pl, cnt, a = full[k]
        assert hist[k][:3] == (me, opp, pl) and hist[k][4] == a
        assert np.array_equal(hist[k][3], mr.policy_from_counts(cnt))
    cells = size * size
    me_h, opp_h, pl_h = hist[h][:3]
    assert cells - bin(me_h | opp_h).count("1") <= empties
    assert cells - bin(hist[h - 1][0] | hist[h - 1][1]).count("1") > empties  # the first position at E empties or fewer
    me = np.array([r[0] for r in hist[h:]], np.uint64)
    opp = np.array([r[1] for r in hist[h:]], np.uint64)
    act, val, mv, _ = pe.endgame_solve(me, opp, size)
    for j, r in enumerate(hist[h:]):
        assert r[4] == act[j] and np.array_equal(r[3], ser.solver_pi(mv[j], val[j]))
        assert r[2] * (1 if j % 2 == 0 else -1) == pl_h  # the side to move alternates, passes included
    assert winner == int(np.sign(val[0])) * pl_h


def test_argument_checks_raise_before_touching_the_gpu():
    from betazero_b200 import loop, selfplay

    for size, bad in ((4, 12), (4, -1), (6, 21), (8, 21)):
        with pytest.raises(ValueError, match="endgame_empties"):
            selfplay.BatchedSelfPlay(8, 8, None, board_size=size, endgame_empties=bad)
    assert selfplay.check_endgame_empties(11, 4) == 11 and selfplay.check_endgame_empties(20, 8) == 20
    assert selfplay.check_endgame_empties(0, 8) == 0
    with pytest.raises(ValueError, match="endgame_every"):
        selfplay.BatchedSelfPlay(8, 8, None, endgame_empties=8, endgame_every=0)
    with pytest.raises(ValueError, match="endgame_cap"):
        selfplay.BatchedSelfPlay(8, 8, None, endgame_empties=8, endgame_cap=0)
    a = loop.default_args()
    assert a.endgame_empties == 0 and a.endgame_every == 8
