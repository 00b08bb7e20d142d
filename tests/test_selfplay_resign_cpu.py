"""CPU: the sequential restatement of self-play with resignation (oracle/selfplay_resign_ref.py) against the games
without it, the host-side false-positive rate and calibration (betazero_b200/resign.py) against brute-force loops, the
layout of bz_selfplay_resign_state against the C compiler, and the argument checks."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import mcts_ref as mr
from oracle import pyoracle as po
from oracle import selfplay_endgame_ref as ser
from oracle import selfplay_resign_ref as srr

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "betazero_b200.h")


def _ev(salt):
    return lambda a, b: mr.hash_eval(a, b, salt, 65)


def test_resign_state_layout_matches_the_c_compiler(tmp_path):
    from betazero_b200._lib import SIGNATURES, BzSelfplayResignState

    fields = [n for n, _ in BzSelfplayResignState._fields_]
    prog = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', "int main(void){",
            'printf("%zu\\n", sizeof(bz_selfplay_resign_state));']
    prog += [f'printf("%zu\\n", offsetof(bz_selfplay_resign_state, {f}));' for f in fields]
    prog += ["return 0;}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(prog))
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-o", str(exe), str(src)])
    vals = [int(v) for v in subprocess.check_output([str(exe)], text=True).split()]
    assert vals == [C.sizeof(BzSelfplayResignState)] + [getattr(BzSelfplayResignState, f).offset for f in fields]
    assert vals[0] == 48 and fields[:BzSelfplayResignState.N_SCALARS] == ["threshold", "reserved", "audit_below"]
    assert "bz_selfplay_advance_resign" in SIGNATURES and "bz_selfplay_endgame_play_resign" in SIGNATURES


@pytest.mark.parametrize("size,n_sims,leaves", [(4, 24, 1), (4, 24, 4), (6, 16, 1), (6, 16, 4)])
def test_never_resigning_is_self_play_game(size, n_sims, leaves):
    """threshold -1, or an audited game: the records are self_play_game's, plus q = W / N of the greedy pick"""
    game = mr.ReversiGame(po.OracleReversiBoard, size)
    full, winner = mr.self_play_game(game, n_sims, 1.25, _ev(3), max_plies=128, leaves=leaves)
    for kw in (dict(threshold=-1.0), dict(threshold=1.0, is_audited=True)):
        hist, w, h, resigned = srr.self_play_game_resign(game, n_sims, 1.25, _ev(3), leaves=leaves, **kw)
        assert w == winner and h is None and not resigned and len(hist) == len(full)
        for r, (me, opp, pl, cnt, a) in zip(hist, full):
            assert r[:3] == (me, opp, pl) and r[4] == a and np.array_equal(r[3], mr.policy_from_counts(cnt))
            assert r[5].dtype == np.float32 and -1 <= r[5] <= 1


@pytest.mark.parametrize("size,n_sims,empties,leaves", [(4, 24, 6, 1), (6, 16, 10, 4)])
def test_never_resigning_with_the_handover_is_the_endgame_restatement(size, n_sims, empties, leaves):
    game = mr.ReversiGame(po.OracleReversiBoard, size)
    solve = ser.c_solver(game)
    ref, winner, h = ser.self_play_game_endgame(game, n_sims, 1.25, _ev(5), empties, solve=solve, leaves=leaves)
    hist, w, h2, resigned = srr.self_play_game_resign(game, n_sims, 1.25, _ev(5), -1.0, endgame_empties=empties,
                                                      solve=solve, leaves=leaves)
    assert (w, h2, resigned) == (winner, h, False) and h is not None and len(hist) == len(ref)
    for k, (r, x) in enumerate(zip(hist, ref)):
        assert r[:3] == x[:3] and r[4] == x[4] and np.array_equal(r[3], x[3])
        assert np.isnan(r[5]) == (k >= h)  # solver-played records carry q = NaN


def _first_low_after(q, start):
    """a ply r >= start whose q is a new running minimum, and a threshold v with q_r < v <= every earlier q"""
    qe = np.asarray(q, np.float32)
    for r in range(max(start, 1), len(qe)):
        lo = qe[:r].min()
        if qe[r] < lo:
            return r, np.nextafter(qe[r], np.float32(np.inf), dtype=np.float32)
    return None, None


@pytest.mark.parametrize("size,n_sims,leaves", [(4, 24, 1), (4, 24, 4), (6, 16, 1), (6, 16, 4), (8, 16, 1), (8, 16, 4)])
def test_a_threshold_from_the_q_trace_ends_the_game_at_its_first_ply_below(size, n_sims, leaves):
    game = mr.ReversiGame(po.OracleReversiBoard, size)
    salt = 7
    full, winner, _, _ = srr.self_play_game_resign(game, n_sims, 1.25, _ev(salt), -1.0, leaves=leaves)
    q = [r[5] for r in full]
    r, v = _first_low_after(q, 2)
    assert r is not None
    hist, w, h, resigned = srr.self_play_game_resign(game, n_sims, 1.25, _ev(salt), float(v), leaves=leaves)
    assert resigned and h is None and len(hist) == r + 1
    assert w == -hist[r][2]  # the mover of the resigning ply loses
    for a, b in zip(hist, full):
        assert a[:3] == b[:3] and a[4] == b[4] and np.array_equal(a[3], b[3]) and a[5] == b[5]
    z = [w * rec[2] for rec in hist]
    assert z[-1] == -1 and all(zz == (-1 if (len(z) - 1 - k) % 2 == 0 else 1) for k, zz in enumerate(z))
    # the same threshold on an audited game: no resignation
    again, w2, _, res2 = srr.self_play_game_resign(game, n_sims, 1.25, _ev(salt), float(v), is_audited=True,
                                                   leaves=leaves)
    assert not res2 and w2 == winner and len(again) == len(full)


def test_root_q_is_the_greedy_edge_with_one_rounded_division():
    cnt = np.zeros(65, np.int32)
    W = np.zeros(65, np.float32)
    assert np.isnan(srr.root_q(cnt, W))
    cnt[[3, 9, 20]] = [5, 7, 7]
    W[[3, 9, 20]] = [4.0, np.float32(-1.3), np.float32(2.2)]
    assert srr.root_q(cnt, W) == np.float32(-1.3) / np.float32(7)  # the tie goes to the lower action id


def test_audit_draw_and_fraction():
    from betazero_b200 import resign

    assert resign.audit_below(0.0) == 0 and resign.audit_below(1.0) == 1 << 32 and resign.audit_below(0.5) == 1 << 31
    assert srr.audit_below(0.1) == resign.audit_below(0.1) == int(0.1 * 2 ** 32)
    for bad in (-0.1, 1.5, float("nan")):
        with pytest.raises(ValueError, match="resign_audit"):
            resign.audit_below(bad)
    got = [srr.audited(11, g, srr.audit_below(0.3)) for g in range(2000)]
    assert 0.25 < np.mean(got) < 0.35
    assert all(srr.audited(11, g, 1 << 32) for g in range(50)) and not any(srr.audited(11, g, 0) for g in range(50))


# -- false positives and calibration -------------------------------------------------------------------------------------
def _records(games, audited):
    """a replay dict (shuffled record order) from per-game (q, z) lists"""
    rows = [(g, k, q[k], z[k], audited[g]) for g, (q, z) in enumerate(games) for k in range(len(q))]
    rng = np.random.default_rng(0)
    rows = [rows[i] for i in rng.permutation(len(rows))]
    return {"game": np.array([r[0] for r in rows], np.int64), "ply": np.array([r[1] for r in rows], np.int16),
            "q": np.array([r[2] for r in rows], np.float32), "z": np.array([r[3] for r in rows], np.int8),
            "audited": np.array([r[4] for r in rows], bool)}


def _synthetic(n_games, seed):
    rng = np.random.default_rng(seed)
    games = []
    for _ in range(n_games):
        n = int(rng.integers(1, 30))
        q = np.round(rng.uniform(-1, 1, n), 2).astype(np.float32)  # rounded: ties between games and records
        q[rng.random(n) < 0.1] = np.nan
        winner = int(rng.integers(-1, 2))
        z = np.array([winner * (1 if k % 2 == 0 else -1) for k in range(n)], np.int8)
        games.append((q, z))
    return games


def _brute(games, audited, v):
    return srr.false_positive_rate([g for g, a in zip(games, audited) if a], v)


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_false_positive_rate_and_calibrate_against_brute_force(seed):
    from betazero_b200 import resign

    games = _synthetic(80, seed)
    audited = list(np.random.default_rng(seed + 10).random(len(games)) < 0.6)
    rec = _records(games, audited)
    aud = [g for g, a in zip(games, audited) if a]
    assert resign.audited_games(rec) == len(aud)
    for v in [-1.0, -0.5, 0.0, 0.3, 1.0] + [float(x) for x in np.unique(rec["q"][~np.isnan(rec["q"])])[::7]]:
        assert resign.false_positive_rate(rec, v) == _brute(games, audited, v), v
    fps = [srr.false_positive_rate(aud, u) for u in sorted({np.float32(-1)} | {x for q, _ in aud for x in q if x == x})]
    assert any(b < a for a, b in zip(fps, fps[1:]))  # FP is not monotone in v here
    for target in (0.0, 0.02, 0.05, 0.1, 0.2, 0.5, 1.0):
        assert resign.calibrate(rec, target) == srr.calibrate(aud, target, keep=-1.0), target


def test_calibrate_takes_the_prefix_where_fp_is_not_monotone():
    from betazero_b200 import resign

    # game 0's would-be resigner is its ply-1 mover, who won, for v in (0.4, 0.6], and its ply-0 mover, who lost, above;
    # game 1's only record (a loser) resigns above 0.9.  Candidates -1, 0.4, 0.6, 0.9: FP = 0, 0, 1/2, 0
    games = [(np.float32([0.6, 0.4]), np.int8([-1, 1])), (np.float32([0.9]), np.int8([-1]))]
    rec = _records(games, [True, True])
    assert [resign.false_positive_rate(rec, v) for v in (-1, 0.4, 0.6, 0.9, 0.95)] == [0.0, 0.0, 0.5, 0.0, 0.0]
    assert resign.calibrate(rec, 0.0) == float(np.float32(0.4))  # not 0.9: the prefix stops at 0.6
    assert resign.calibrate(rec, 0.5) == float(np.float32(0.9))
    assert srr.calibrate(games, 0.0, keep=-1.0) == resign.calibrate(rec, 0.0)


def test_no_audited_games_keep_the_threshold():
    from betazero_b200 import resign

    games = _synthetic(10, 4)
    rec = _records(games, [False] * len(games))
    assert resign.false_positive_rate(rec, 0.5) == 0.0 and resign.audited_games(rec) == 0
    assert resign.calibrate(rec, 0.05, keep=-0.7) == -0.7 and srr.calibrate([], 0.05, keep=-0.7) == -0.7
    empty = {k: v[:0] for k, v in rec.items()}
    assert resign.calibrate(empty, 0.05, keep=0.25) == 0.25
    with pytest.raises(ValueError, match="target"):
        resign.calibrate(rec, -0.1)


def test_calibrate_on_restated_games():
    """records of restated audited games (hash evaluator) calibrate like the brute-force definition"""
    from betazero_b200 import resign

    games = []
    for salt in range(6):
        game = mr.ReversiGame(po.OracleReversiBoard, 4)
        hist, w, _, _ = srr.self_play_game_resign(game, 16, 1.25, _ev(salt), -1.0)
        games.append((np.array([r[5] for r in hist], np.float32), np.array([w * r[2] for r in hist], np.int8)))
    rec = _records(games, [True] * len(games))
    for target in (0.0, 0.2, 0.5):
        assert resign.calibrate(rec, target) == srr.calibrate(games, target, keep=-1.0)
    for v in (-0.5, 0.0, 0.5):
        assert resign.false_positive_rate(rec, v) == srr.false_positive_rate(games, v)


def test_argument_checks_raise_before_touching_the_gpu():
    from betazero_b200 import loop, resign, selfplay

    for bad in (1.5, -1.01, float("nan")):
        with pytest.raises(ValueError, match="resign threshold"):
            selfplay.BatchedSelfPlay(8, 8, None, resign_threshold=bad)
        with pytest.raises(ValueError, match="resign threshold"):
            resign.check_threshold(bad)
    with pytest.raises(ValueError, match="resign_audit"):
        selfplay.BatchedSelfPlay(8, 8, None, resign_threshold=0.0, resign_audit=2.0)
    assert resign.check_threshold(-1) == -1.0 and resign.check_threshold(0.1) == float(np.float32(0.1))
    a = loop.default_args()
    assert a.resign is None and a.resign_audit == 0.1 and a.resign_fp is None


def _dist_worker(rank, world, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    import torch
    import torch.distributed as dist

    from betazero_b200 import dist as bzd
    from betazero_b200 import resign

    bzd.init("gloo")
    games = _synthetic(40, 20 + rank)  # each rank's shard: its own games, ids rank*40 + g
    audited = list(np.random.default_rng(30 + rank).random(len(games)) < 0.5)
    rec = _records(games, audited)
    shard = {"game": torch.from_numpy(rec["game"] + 40 * rank), "ply": torch.from_numpy(rec["ply"]),
             "q": torch.from_numpy(rec["q"]), "z": torch.from_numpy(rec["z"]),
             "audited": torch.from_numpy(rec["audited"])}
    allr = bzd.gather_replay(shard)
    ret[rank] = {"v": resign.calibrate(allr, 0.1, keep=-1.0), "fp": resign.false_positive_rate(allr, 0.0),
                 "n": int(allr["game"].numel())}
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.timeout(120)
def test_world_size_2_gloo_ranks_calibrate_the_same_threshold():
    import socket

    import torch.multiprocessing as mp

    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ret = mp.Manager().dict()
    mp.spawn(_dist_worker, args=(2, port, ret), nprocs=2, join=True)
    r0, r1 = ret[0], ret[1]
    assert r0 == r1
    games = _synthetic(40, 20) + _synthetic(40, 21)
    audited = list(np.random.default_rng(30).random(40) < 0.5) + list(np.random.default_rng(31).random(40) < 0.5)
    aud = [g for g, a in zip(games, audited) if a]
    assert r0["n"] == sum(len(q) for q, _ in games)
    assert r0["v"] == srr.calibrate(aud, 0.1, keep=-1.0) and r0["fp"] == srr.false_positive_rate(aud, 0.0)
