"""GPU: self-play with the endgame handover (BatchedSelfPlay(endgame_empties=E); bz_selfplay_advance_endgame,
bz_selfplay_endgame_play) against the sequential restatement (oracle/selfplay_endgame_ref.py), the records of the same
games without the feature, the exact solver, and across solver schedules, queue overflow, tree reuse and the one-launch
search."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import mcts_ref as mr  # noqa: E402
from oracle import pyoracle as po  # noqa: E402
from oracle import selfplay_endgame_ref as ser  # noqa: E402

pytestmark = pytest.mark.gpu


def _games(rp):
    """game id -> (me, opp, pi, z) in ply order; every game's plies are 0 .. n-1"""
    game, ply = rp["game"].cpu().numpy(), rp["ply"].cpu().numpy()
    me, opp = rp["me"].cpu().numpy().view(np.uint64), rp["opp"].cpu().numpy().view(np.uint64)
    pi, z = rp["pi"].cpu().numpy(), rp["z"].cpu().numpy()
    out = {}
    order = np.lexsort((ply, game))
    bounds = np.flatnonzero(np.diff(game[order])) + 1
    for idx in np.split(order, bounds):
        if idx.size == 0:
            continue
        assert np.array_equal(ply[idx], np.arange(idx.size))
        out[int(game[idx[0]])] = (me[idx], opp[idx], pi[idx], z[idx])
    return out


def _empties(me, opp, size):
    return size * size - np.array([bin(int(m) | int(o)).count("1") for m, o in zip(me, opp)])


def _check_against_feature_off(on, off, size, empties, min_common):
    """every game finished in both runs: identical records before the handover (all of them without one); the records
    from the handover on are perfect play: pi uniform over the optimal moves, z the sign of the exact value for the
    record's mover, which is also the z of the searched prefix (the side to move alternates every ply)"""
    from betazero_b200 import env, minimax

    common = sorted(set(on) & set(off))
    assert len(common) >= min_common
    boards, where, handed = [], [], 0
    for g in common:
        me, opp, pi, z = on[g]
        e = _empties(me, opp, size)
        h = int(np.argmax(e <= empties)) if (e <= empties).any() else len(me)  # the start position is always searched
        ome, oopp, opi, oz = off[g]
        assert np.array_equal(me[:h], ome[:h]) and np.array_equal(opp[:h], oopp[:h]) and np.array_equal(pi[:h], opi[:h]), g
        if h == len(me):
            assert len(me) == len(ome) and np.array_equal(z, oz), g
            continue
        handed += 1
        sign = np.where(np.arange(len(me)) % 2 == h % 2, 1, -1)
        assert np.array_equal(z, z[h] * sign), g
        boards.append((me[h:], opp[h:], pi[h:], z[h:]))
    assert handed >= min_common // 2
    me = np.concatenate([b[0] for b in boards])
    opp = np.concatenate([b[1] for b in boards])
    act, val, mv, _ = minimax.solve(env.to_device_u64(me), env.to_device_u64(opp), size)
    val, mv = val.cpu().numpy(), mv.cpu().numpy()
    pi = np.concatenate([b[2] for b in boards])
    z = np.concatenate([b[3] for b in boards])
    assert np.array_equal(z, np.sign(val).astype(np.int8))
    for j in range(len(me)):
        assert np.array_equal(pi[j], ser.solver_pi(mv[j], val[j])), j
    return handed


@pytest.mark.parametrize("size,n_sims,empties,leaves", [(4, 24, 6, 1), (4, 24, 6, 4), (6, 16, 10, 1), (6, 16, 10, 4),
                                                       (8, 32, 8, 1), (8, 32, 8, 4), (8, 32, 12, 1), (8, 32, 12, 4)])
def test_deterministic_handover_equals_sequential_restatement(size, n_sims, empties, leaves):
    """temp_plies = 0: every slot plays the restatement's game; actions, records, z, counters, restarts and game ids"""
    from betazero_b200 import mcts, selfplay

    salt = 3
    game = mr.ReversiGame(po.OracleReversiBoard, size)
    hist, winner, h = ser.self_play_game_endgame(game, n_sims, 1.25, lambda a, b: mr.hash_eval(a, b, salt, 65), empties,
                                                 solve=ser.c_solver(game), leaves=leaves)
    assert h is not None
    B = 5
    sp = selfplay.BatchedSelfPlay(B, n_sims, mcts.HashEvaluator(salt), board_size=size, temp_plies=0, use_graph=False,
                                  rank=1, world=3, n_leaves=leaves, endgame_empties=empties, endgame_every=1)
    for ply in range(h):
        assert sp.ply.tolist() == [ply] * B and sp.game_id.tolist() == [5, 6, 7, 8, 9]
        sp.play_move()
        assert sp.last_action.tolist() == [hist[ply][4]] * B
    sp.mcts.check_errors()
    st = sp.stats()
    n = len(hist)
    assert st["games"] == B and st["plies"] == B * n and st["replay_records"] == B * n and st["dropped"] == 0
    assert st[{1: "x_wins", -1: "o_wins", 0: "draws"}[winner]] == B
    assert st["endgame_games"] == B and st["endgame_plies"] == B * (n - h)
    assert st["endgame_pending"] == 0 and st["endgame_overflow"] == 0
    assert sp.ply.tolist() == [0] * B and sp.player.tolist() == [1] * B
    assert sp.game_id.tolist() == [20, 21, 22, 23, 24]  # id_stride = world * B
    assert sp.eg_counters[0].item() == B  # handed over
    got = _games(sp.drain_replay())
    assert sorted(got) == [5, 6, 7, 8, 9]
    for g in got:
        me, opp, pi, z = got[g]
        assert len(me) == n
        for k, (hme, hopp, hpl, hpi, _) in enumerate(hist):
            assert me[k] == hme and opp[k] == hopp and z[k] == winner * hpl and np.array_equal(pi[k], hpi), (g, k)


def _run(B, n_sims, plies, size=8, **kw):
    from betazero_b200 import mcts, selfplay

    sp = selfplay.BatchedSelfPlay(B, n_sims, kw.pop("evaluator", None) or mcts.HashEvaluator(7), board_size=size,
                                  use_graph=False, **kw)
    for _ in range(plies):
        sp.play_move()
    sp.mcts.check_errors()
    return sp


def test_prefix_identity_and_perfect_endgames_with_sampled_moves():
    kw = dict(temp_plies=24, seed=11)
    off = _run(128, 16, 140, **kw)
    on = _run(128, 16, 140, endgame_empties=8, **kw)
    st = on.stats()
    assert st["endgame_overflow"] == 0 and st["endgame_games"] > 128 and st["dropped"] == 0
    _check_against_feature_off(_games(on.drain_replay()), _games(off.drain_replay()), 8, 8, min_common=128)


def test_solver_schedule_does_not_change_the_records():
    # a slot reaches 10 empties ~22 plies after a restart, so 32 plies can hand over two games per slot: a queue of 2 B
    runs = [_run(64, 16, 100, size=6, temp_plies=10, seed=4, endgame_empties=10, endgame_every=k, endgame_cap=128)
            for k in (1, 8, 32)]
    assert all(sp.stats()["endgame_overflow"] == 0 for sp in runs)
    games = [_games(sp.drain_replay()) for sp in runs]
    common = set(games[0]) & set(games[1]) & set(games[2])
    assert len(common) >= 64
    for g in common:
        for other in games[1:]:
            assert all(np.array_equal(a, b) for a, b in zip(games[0][g], other[g])), g
    # the slots restart at the handover whatever the schedule: the same games are in progress
    assert runs[0].game_id.tolist() == runs[1].game_id.tolist() == runs[2].game_id.tolist()


def test_queue_overflow_keeps_games_in_their_slots():
    """a tiny queue: the games that do not fit are searched to their end and counted; every record is still valid, and a
    full replay buffer still drops whole games"""
    kw = dict(size=4, temp_plies=30, seed=3)
    off = _run(48, 8, 40, **kw)
    on = _run(48, 8, 40, endgame_empties=6, endgame_cap=2, **kw)
    st = on.stats()
    assert st["endgame_overflow"] > 0 and st["endgame_games"] > 0
    assert st["games"] == st["x_wins"] + st["o_wins"] + st["draws"]
    rp = on.drain_replay()
    me, opp = rp["me"].cpu().numpy().view(np.uint64), rp["opp"].cpu().numpy().view(np.uint64)
    pi = rp["pi"].cpu().numpy()
    assert not (me & opp).any()
    np.testing.assert_allclose(pi.sum(1), 1.0, atol=1e-5)
    mask = po.legal_mask(me, opp, 4)
    legal = ((mask[:, None] >> np.arange(64, dtype=np.uint64)) & np.uint64(1)).astype(bool)
    assert (pi[:, :64][~legal] == 0).all() and ((pi[:, 64] > 0) == (mask == 0)).all()
    got, ref = _games(rp), _games(off.drain_replay())
    same = [g for g in set(got) & set(ref) if len(got[g][0]) == len(ref[g][0])
            and all(np.array_equal(a, b) for a, b in zip(got[g], ref[g]))]
    assert len(same) > 0  # refused games (and those that end before E empties) are the games without the feature

    small = _run(48, 8, 14, endgame_empties=6, endgame_every=2, replay_cap=100, **kw)
    st = small.stats()
    assert st["dropped"] > 0 and st["replay_records"] <= 100
    with pytest.warns(RuntimeWarning, match="replay buffer overflow"):
        got = _games(small.drain_replay())
    assert 0 < sum(len(v[0]) for v in got.values()) <= 100


def test_reuse_restarts_handed_over_slots_with_empty_trees():
    """reuse=True, deterministic moves: the game that follows a handover in a slot starts from an empty tree, so it is
    the same game again, and its records equal those of reuse=True without the feature up to the handover"""
    from betazero_b200 import mcts, selfplay

    size, n_sims, E, B = 6, 16, 10, 4
    mk = lambda **k: selfplay.BatchedSelfPlay(B, n_sims, mcts.HashEvaluator(5), board_size=size, temp_plies=0,  # noqa: E731
                                              use_graph=False, reuse=True, **k)
    off = mk()
    for _ in range(40):
        off.play_move()
    on = mk(endgame_empties=E, endgame_every=1)
    gid0 = on.game_id.tolist()
    for _ in range(100):
        if on.stats()["endgame_games"] >= 2 * B:
            break
        on.play_move()
    assert on.stats()["endgame_overflow"] == 0
    got, ref = _games(on.drain_replay()), _games(off.drain_replay())
    first = got[gid0[0]]
    h = int(np.argmax(_empties(first[0], first[1], size) <= E))
    assert h > 0
    for g, recs in got.items():
        assert all(np.array_equal(a, b) for a, b in zip(recs, first)), g
    r = ref[gid0[0]]
    assert all(np.array_equal(a[:h], b[:h]) for a, b in zip(first[:3], r[:3]))


def test_one_launch_search_and_the_bf16_net():
    from betazero_b200 import mcts, net

    model = net.make_net("mlp", seed=2)
    kw = dict(temp_plies=60, seed=5, n_leaves=4)
    off = _run(256, 16, 90, evaluator=mcts.FusedNetEvaluator(model), **kw)
    on = _run(256, 16, 90, evaluator=mcts.FusedNetEvaluator(model), endgame_empties=8, **kw)
    assert on.mcts.one_launch
    _check_against_feature_off(_games(on.drain_replay()), _games(off.drain_replay()), 8, 8, min_common=128)


def test_off_means_off():
    """endgame_empties = 0 launches what self-play launches without the option and gives the same records"""
    kw = dict(size=4, temp_plies=20, seed=9)
    a = _run(32, 8, 30, **kw)
    b = _run(32, 8, 30, endgame_empties=0, endgame_every=1, **kw)
    assert b.eg is None and a.total_launches() == b.total_launches()
    sa, sb = a.stats(), b.stats()
    assert sa == sb and sb["endgame_games"] == sb["endgame_plies"] == sb["endgame_pending"] == sb["endgame_overflow"] == 0
    ga, gb = _games(a.drain_replay()), _games(b.drain_replay())
    assert sorted(ga) == sorted(gb) and all(all(np.array_equal(x, y) for x, y in zip(ga[g], gb[g])) for g in ga)


def test_refusals():
    from betazero_b200 import _lib, mcts, selfplay

    sp = selfplay.BatchedSelfPlay(8, 8, mcts.HashEvaluator(1), board_size=6, endgame_empties=10, use_graph=False)
    L = _lib.load()
    sp.search()
    eg = sp.eg
    for field, bad in (("empties", 0), ("empties", 32), ("cap", 0), ("max_plies", 64)):
        old = getattr(eg, field)
        setattr(eg, field, bad)
        assert L.bz_selfplay_advance_endgame(sp._ref, sp._eg_ref, sp.pools._ref, None, _lib.stream_ptr()) == -1, field
        assert L.bz_selfplay_endgame_play(sp._ref, sp._eg_ref, _lib.dptr(sp.eg_workspace), _lib.stream_ptr()) == -1
        setattr(eg, field, old)
    assert L.bz_selfplay_endgame_play(sp._ref, sp._eg_ref, None, _lib.stream_ptr()) == -1
    assert L.bz_selfplay_endgame_play(sp._ref, sp._eg_ref, C_offset(sp.eg_workspace, 4), _lib.stream_ptr()) == -2
    assert L.bz_selfplay_endgame_workspace_bytes(0) == 0


def C_offset(t, k):
    import ctypes

    return ctypes.c_void_p(t.data_ptr() + k)


def test_loop_reports_the_endgame_entry():
    import math

    from betazero_b200 import loop

    args = loop.default_args(games=256, sims=16, leaves=4, plies=70, train_steps=2, batch=256, lr=1e-3,
                             endgame_empties=8, endgame_every=8)
    (line,) = loop.run(args)
    e = line["endgame"]
    assert e["empties"] == 8 and e["every"] == 8 and e["games"] > 0 and e["plies"] > 0 and e["ms"] > 0
    assert e["overflow"] == 0 and e["pending"] >= 0
    assert line["replay_records_gathered"] > 0 and all(math.isfinite(x) for x in line["loss_first_last"])
    assert "endgame" not in loop.run_iteration(loop.LoopState(loop.default_args(games=48, sims=16, plies=2, size=6,
                                                                                train_steps=1, batch=64), 0, 1), 0)
