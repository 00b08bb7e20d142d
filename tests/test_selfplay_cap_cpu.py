"""CPU: the sequential restatement of self-play with randomized search budgets (oracle/selfplay_cap_ref.py) against the
games without them (mcts_ref.self_play_game, selfplay_resign_ref.self_play_game_resign) for the identities p = 1 and
fast_sims == n_sims, the full-ply draw, the layout of bz_selfplay_cap_state against the C compiler, and the argument
checks."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import mcts_ref as mr
from oracle import pyoracle as po
from oracle import selfplay_cap_ref as scr
from oracle import selfplay_endgame_ref as ser
from oracle import selfplay_resign_ref as srr
from oracle.minimax_ref import philox_u32

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "betazero_b200.h")
ALL = 1 << 32


def _ev(salt):
    return lambda a, b: mr.hash_eval(a, b, salt, 65)


def test_cap_state_layout_matches_the_c_compiler(tmp_path):
    from betazero_b200._lib import SIGNATURES, BzSelfplayCapState

    fields = [n for n, _ in BzSelfplayCapState._fields_]
    prog = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', "int main(void){",
            'printf("%zu\\n", sizeof(bz_selfplay_cap_state));']
    prog += [f'printf("%zu\\n", offsetof(bz_selfplay_cap_state, {f}));' for f in fields]
    prog += ["return 0;}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(prog))
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-o", str(exe), str(src)])
    vals = [int(v) for v in subprocess.check_output([str(exe)], text=True).split()]
    assert vals == [C.sizeof(BzSelfplayCapState)] + [getattr(BzSelfplayCapState, f).offset for f in fields]
    assert vals[0] == 80 and fields[:BzSelfplayCapState.N_SCALARS] == ["full_below", "n_trees", "reserved"]
    for name in ("bz_selfplay_cap_layout", "bz_selfplay_advance_cap", "bz_selfplay_endgame_play_cap",
                 "bz_mcts_root_noise_entrant"):
        assert name in SIGNATURES


def test_the_draw_is_philox_on_its_own_counter():
    from betazero_b200 import selfplay

    assert scr.full_below(0.25) == selfplay.full_below(0.25) == 1 << 30
    assert selfplay.full_below(0.0) == 0 and selfplay.full_below(1.0) == ALL and selfplay.FULL_COUNTER == scr.FULL_COUNTER
    below = scr.full_below(0.3)
    draws = [(g, t) for g in range(40) for t in range(60)]
    got = np.array([scr.is_full(11, g, t, below) for g, t in draws])
    assert got.tolist() == [philox_u32(11, g, 0x80000000 | t) < below for g, t in draws]
    assert 0.26 < got.mean() < 0.34
    # not the move-sampling draw (counter t) and not the resignation audit's (counter 0xFFFFFFFF)
    assert any(philox_u32(11, g, 0x80000000 | t) != philox_u32(11, g, t) for g, t in draws[:5])
    assert all(0x80000000 | t not in (t, srr.AUDIT_COUNTER) for t in range(128))
    assert all(scr.is_full(3, g, t, ALL) for g, t in draws[:50]) and not any(scr.is_full(3, g, t, 0) for g, t in draws[:50])


def test_sampled_move_is_the_first_prefix_above_the_target():
    cnt = np.zeros(65, np.int32)
    cnt[[2, 7, 30, 64]] = [3, 0, 5, 2]
    for g in range(200):
        r = philox_u32(5, g, 3)
        target = (r * 10) >> 32
        cum, want = 0, None
        for a in range(65):
            cum += int(cnt[a])
            if cum > target:
                want = a
                break
        assert scr.sampled_move(cnt, 5, g, 3) == want


@pytest.mark.parametrize("size,n_sims,leaves", [(4, 24, 1), (4, 24, 4), (6, 16, 1), (6, 16, 4)])
def test_every_ply_full_is_self_play_game(size, n_sims, leaves):
    """p = 1: the records of self_play_game, every flag 1, whatever fast_sims is"""
    game = mr.ReversiGame(po.OracleReversiBoard, size)
    full, winner = mr.self_play_game(game, n_sims, 1.25, _ev(3), max_plies=128, leaves=leaves)
    search = scr.mcts_search(game, 1.25, _ev(3), leaves)
    hist, w, h, resigned = scr.self_play_game_cap(game, n_sims, 2 * leaves, search, 7, 12, ALL)
    assert (w, h, resigned) == (winner, None, False) and len(hist) == len(full)
    for r, (me, opp, pl, cnt, a) in zip(hist, full):
        assert r[:3] == (me, opp, pl) and r[4] == a and np.array_equal(r[3], mr.policy_from_counts(cnt)) and r[6] == 1


@pytest.mark.parametrize("size,n_sims,leaves,p", [(4, 24, 1, 0.3), (6, 16, 4, 0.5), (6, 16, 1, 0.0)])
def test_equal_budgets_are_self_play_game_with_the_flags_of_the_draw(size, n_sims, leaves, p):
    game = mr.ReversiGame(po.OracleReversiBoard, size)
    full, winner = mr.self_play_game(game, n_sims, 1.25, _ev(4), max_plies=128, leaves=leaves)
    search = scr.mcts_search(game, 1.25, _ev(4), leaves)
    below = scr.full_below(p)
    hist, w, _, _ = scr.self_play_game_cap(game, n_sims, n_sims, search, 9, 31, below)
    assert w == winner and len(hist) == len(full)
    for t, (r, (me, opp, pl, cnt, a)) in enumerate(zip(hist, full)):
        assert r[:3] == (me, opp, pl) and r[4] == a and np.array_equal(r[3], mr.policy_from_counts(cnt))
        assert r[6] == int(philox_u32(9, 31, 0x80000000 | t) < below)


@pytest.mark.parametrize("size,n_sims,fast,leaves", [(4, 24, 8, 1), (6, 32, 8, 4), (8, 16, 4, 1)])
def test_each_ply_is_searched_at_the_budget_of_its_flag(size, n_sims, fast, leaves):
    game = mr.ReversiGame(po.OracleReversiBoard, size)
    search = scr.mcts_search(game, 1.25, _ev(6), leaves)
    below = scr.full_below(0.4)
    hist, _, _, _ = scr.self_play_game_cap(game, n_sims, fast, search, 2, 77, below)
    flags = [r[6] for r in hist]
    assert 0 < sum(flags) < len(flags)
    board, player = game.initial()
    for t, r in enumerate(hist):
        assert game.wire(board, player) == r[:2] and player == r[2]
        cnt, _ = search(board, player, n_sims if r[6] else fast)
        assert np.array_equal(r[3], mr.policy_from_counts(cnt)) and r[4] == mr.pick_move(cnt), t
        board, player = game.next(board, player, r[4])
    # the budgets matter: the same game with every ply full differs
    again, _, _, _ = scr.self_play_game_cap(game, n_sims, fast, search, 2, 77, ALL)
    assert [r[4] for r in again] != [r[4] for r in hist] or any(not np.array_equal(a[3], b[3]) for a, b in zip(again, hist))


@pytest.mark.parametrize("size,n_sims,empties,leaves", [(4, 24, 6, 1), (6, 16, 10, 4)])
def test_with_resignation_and_the_handover_it_is_the_resign_restatement(size, n_sims, empties, leaves):
    """p = 1 (and fast_sims == n_sims at p = 0.5): self_play_game_resign's records, the solver's records full"""
    game = mr.ReversiGame(po.OracleReversiBoard, size)
    solve = ser.c_solver(game)
    search = scr.mcts_search(game, 1.25, _ev(5), leaves)
    ref, winner, h, _ = srr.self_play_game_resign(game, n_sims, 1.25, _ev(5), -1.0, endgame_empties=empties, solve=solve,
                                                  leaves=leaves)
    assert h is not None
    for fast, below in ((2 * leaves, ALL), (n_sims, scr.full_below(0.5))):
        hist, w, h2, resigned = scr.self_play_game_cap(game, n_sims, fast, search, 4, 8, below, threshold=-1.0,
                                                       endgame_empties=empties, solve=solve)
        assert (w, h2, resigned) == (winner, h, False) and len(hist) == len(ref)
        for k, (r, x) in enumerate(zip(hist, ref)):
            assert r[:3] == x[:3] and r[4] == x[4] and np.array_equal(r[3], x[3])
            assert np.array_equal(r[5], x[5], equal_nan=True)
            assert r[6] == (1 if k >= h or below == ALL else int(scr.is_full(4, 8, k, below)))
    # a threshold from the q trace resigns at the same ply as the resign restatement
    q = np.array([x[5] for x in ref[:h]], np.float32)
    r = next(k for k in range(2, len(q)) if q[k] < q[:k].min())
    v = float(np.nextafter(q[r], np.float32(np.inf), dtype=np.float32))
    hist, w, _, resigned = scr.self_play_game_cap(game, n_sims, 2 * leaves, search, 4, 8, ALL, threshold=v,
                                                  endgame_empties=empties, solve=solve)
    assert resigned and len(hist) == r + 1 and w == -hist[r][2]


def test_argument_checks_raise_before_touching_the_gpu():
    from betazero_b200 import loop, mcts, selfplay

    class Fake(mcts.FusedNetEvaluator):
        def __init__(self):  # never bound: the checks come first
            pass

    for kw, match in ((dict(fast_sims=8, full_fraction=1.5), "full_fraction"),
                      (dict(fast_sims=8, full_fraction=-0.1), "full_fraction"),
                      (dict(fast_sims=8, full_fraction=float("nan")), "full_fraction"),
                      (dict(fast_sims=4, n_leaves=4), "fast_sims"), (dict(fast_sims=6, n_leaves=4), "fast_sims"),
                      (dict(fast_sims=40), "fast_sims"), (dict(fast_sims=1), "fast_sims"),
                      (dict(fast_sims=8, reuse=True), "tree reuse"), (dict(fast_sims=8, one_launch=False), "one-launch"),
                      (dict(fast_sims=16, n_leaves=8), "one-launch")):
        with pytest.raises(ValueError, match=match):
            selfplay.BatchedSelfPlay(8, 32, Fake(), **kw)
    with pytest.raises(ValueError, match="one-launch"):
        selfplay.BatchedSelfPlay(8, 32, None, fast_sims=8)
    with pytest.raises(ValueError, match="one-launch"):
        selfplay.BatchedSelfPlay(8, 32, mcts.HashEvaluator(1), fast_sims=8)
    assert selfplay.check_fast_sims(8, 32, 4) == 8 and selfplay.check_fast_sims(32, 32, 1) == 32
    a = loop.default_args()
    assert a.fast_sims is None and a.full_fraction == 0.25
