"""GPU: self-play with resignation (BatchedSelfPlay(resign_threshold=v, resign_audit=f); bz_selfplay_advance_resign,
bz_selfplay_endgame_play_resign) against the sequential restatement (oracle/selfplay_resign_ref.py), and against the
same games without resignation: every resigned game is a prefix of its full game up to its first ply with q < v."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import endgame_wld_ref as ewr  # noqa: E402
from oracle import mcts_ref as mr  # noqa: E402
from oracle import pyoracle as po  # noqa: E402
from oracle import selfplay_endgame_ref as ser  # noqa: E402
from oracle import selfplay_resign_ref as srr  # noqa: E402

pytestmark = pytest.mark.gpu


def _games(rp):
    """game id -> (me, opp, pi, z, q) in ply order; every game's plies are 0 .. n-1"""
    game, ply = rp["game"].cpu().numpy(), rp["ply"].cpu().numpy()
    cols = [rp["me"].cpu().numpy().view(np.uint64), rp["opp"].cpu().numpy().view(np.uint64), rp["pi"].cpu().numpy(),
            rp["z"].cpu().numpy()]
    if "q" in rp:
        cols.append(rp["q"].cpu().numpy())
    out = {}
    order = np.lexsort((ply, game))
    for idx in np.split(order, np.flatnonzero(np.diff(game[order])) + 1):
        if idx.size:
            assert np.array_equal(ply[idx], np.arange(idx.size))
            out[int(game[idx[0]])] = tuple(c[idx] for c in cols)
    return out


def _same(a, b):
    return all(np.array_equal(x, y, equal_nan=x.dtype.kind == "f") for x, y in zip(a, b))


def _first_low(q, start=2):
    """a ply r >= start whose q is below every earlier q, and a threshold v with q_r < v <= every earlier q"""
    qe = np.asarray(q, np.float32)
    for r in range(start, len(qe)):
        if qe[r] < qe[:r].min():
            return r, float(np.nextafter(qe[r], np.float32(np.inf), dtype=np.float32))
    return None, None


CASES = [(4, 24, 1, 0, "exact"), (4, 24, 4, 4, "exact"), (4, 24, 1, 6, "wld"), (4, 24, 4, 0, "exact"),
         (6, 16, 1, 0, "exact"), (6, 16, 4, 10, "wld"), (6, 16, 1, 10, "exact"), (6, 16, 4, 0, "exact"),
         (8, 32, 1, 8, "exact"), (8, 32, 4, 0, "exact"), (8, 32, 1, 0, "exact"), (8, 32, 4, 8, "wld")]


@pytest.mark.parametrize("size,n_sims,leaves,empties,solve", CASES)
def test_deterministic_resignation_equals_sequential_restatement(size, n_sims, leaves, empties, solve):
    """temp_plies = 0: every slot plays the restatement's game; actions, records, q, z, counters, restarts, game ids --
    at threshold -1, at a threshold taken from the game's own q trace (it resigns there), and audited (it does not)"""
    from betazero_b200 import mcts, selfplay

    salt = 3
    game = mr.ReversiGame(po.OracleReversiBoard, size)
    ev = lambda a, b: mr.hash_eval(a, b, salt, 65)  # noqa: E731
    solver = ser.c_solver(game) if solve == "exact" else ewr.wld_solver(ser.c_solver(game))
    kw = dict(endgame_empties=empties, solve=solver, leaves=leaves)
    full, _, h, _ = srr.self_play_game_resign(game, n_sims, 1.25, ev, -1.0, **kw)
    assert (h is not None) == (empties > 0)
    r, v = _first_low([rec[5] for rec in full[:h]])
    assert r is not None
    B = 5
    for thr, audit in ((-1.0, 0.0), (v, 0.0), (v, 1.0)):
        hist, winner, hh, resigned = srr.self_play_game_resign(game, n_sims, 1.25, ev, thr, is_audited=audit == 1.0, **kw)
        assert resigned == (thr == v and audit == 0.0)
        sp = selfplay.BatchedSelfPlay(B, n_sims, mcts.HashEvaluator(salt), board_size=size, temp_plies=0, use_graph=False,
                                      rank=1, world=3, n_leaves=leaves, endgame_empties=empties, endgame_every=1,
                                      endgame_solve=solve, resign_threshold=thr, resign_audit=audit)
        searched = hh if hh is not None else len(hist)
        for ply in range(searched):
            assert sp.ply.tolist() == [ply] * B and sp.game_id.tolist() == [5, 6, 7, 8, 9]
            sp.play_move()
            assert sp.last_action.tolist() == [hist[ply][4]] * B
        sp.mcts.check_errors()
        st = sp.stats()
        n = len(hist)
        assert st["games"] == B and st["plies"] == B * n and st["replay_records"] == B * n and st["dropped"] == 0
        assert st[{1: "x_wins", -1: "o_wins", 0: "draws"}[winner]] == B
        assert st["resigned"] == (B if resigned else 0) and st["audited"] == (B if audit == 1.0 else 0)
        assert st["endgame_games"] == (B if hh is not None else 0)
        assert sp.ply.tolist() == [0] * B and sp.player.tolist() == [1] * B
        assert sp.game_id.tolist() == [20, 21, 22, 23, 24]  # id_stride = world * B
        got = _games(sp.drain_replay())
        assert sorted(got) == [5, 6, 7, 8, 9]
        for g, (me, opp, pi, z, q) in got.items():
            assert len(me) == n
            for k, (hme, hopp, hpl, hpi, _, hq) in enumerate(hist):
                assert me[k] == hme and opp[k] == hopp and z[k] == winner * hpl and np.array_equal(pi[k], hpi), (g, k)
                assert np.array_equal(q[k], hq, equal_nan=True), (g, k, q[k], hq)


def _run(B, n_sims, plies, size=8, **kw):
    from betazero_b200 import mcts, selfplay

    sp = selfplay.BatchedSelfPlay(B, n_sims, kw.pop("evaluator", None) or mcts.HashEvaluator(7), board_size=size,
                                  use_graph=False, **kw)
    for _ in range(plies):
        sp.play_move()
    sp.mcts.check_errors()
    return sp


def _check_prefixes(on, full, v, audited=frozenset(), min_common=64):
    """every game finished in both runs: an audited game, or one whose q never falls below v, is its full game; any
    other game is the full game's prefix up to its first q < v, and its mover there lost"""
    common = sorted(set(on) & set(full))
    assert len(common) >= min_common
    resigned = 0
    for g in common:
        rec, ref = on[g], full[g]
        below = np.flatnonzero(ref[4] < np.float32(v))
        if g in audited or below.size == 0:
            assert len(rec[0]) == len(ref[0]) and _same(rec, ref), g
            continue
        r = int(below[0])
        resigned += 1
        assert len(rec[0]) == r + 1 and _same([x[:r + 1] for x in rec[:3]] + [rec[4]], [x[:r + 1] for x in ref[:3]] +
                                              [ref[4][:r + 1]]), g
        assert np.array_equal(rec[3], np.where((r - np.arange(r + 1)) % 2 == 0, -1, 1).astype(np.int8)), g
    return resigned


def test_sampled_moves_audit_all_threshold_and_half_audited():
    from betazero_b200 import resign

    kw = dict(temp_plies=24, seed=11)
    off = _run(128, 16, 140, **kw)
    every = _run(128, 16, 140, resign_threshold=0.5, resign_audit=1.0, **kw)
    st = every.stats()
    assert st["resigned"] == 0 and st["audited"] == st["games"] > 128
    g_off, g_all = _games(off.drain_replay()), _games(every.drain_replay())
    assert sorted(g_off) == sorted(g_all)
    for g in g_off:
        assert _same(g_all[g][:4], g_off[g]) and not np.isnan(g_all[g][4]).any(), g
    q = np.concatenate([x[4] for x in g_all.values()])
    assert ((q >= -1) & (q <= 1)).all()
    v = float(np.float32(np.quantile(q, 0.05)))
    on = _run(128, 16, 140, resign_threshold=v, resign_audit=0.0, **kw)
    assert on.stats()["resigned"] > 0 and on.stats()["audited"] == 0
    assert _check_prefixes(_games(on.drain_replay()), g_all, v) > 16
    half = _run(128, 16, 140, resign_threshold=v, resign_audit=0.5, **kw)
    got = _games(half.drain_replay())
    ids = torch.tensor(sorted(got), dtype=torch.int64, device="cuda")
    aud = {int(g) for g, a in zip(ids.tolist(), resign.audited(ids, 11, 0.5).tolist()) if a}
    assert 0.3 < len(aud) / len(got) < 0.7
    st = half.stats()
    assert st["resigned"] > 0 and st["audited"] >= len(aud)
    assert _check_prefixes(got, g_all, v, audited=aud) > 8


@pytest.mark.parametrize("reuse", [False, True])
def test_one_launch_search_and_the_bf16_net(reuse):
    from betazero_b200 import mcts, net

    model = net.make_net("mlp", seed=2)
    kw = dict(temp_plies=60, seed=5, n_leaves=4, reuse=reuse)
    every = _run(512, 16, 90, evaluator=mcts.FusedNetEvaluator(model), resign_threshold=1.0, resign_audit=1.0, **kw)
    assert every.mcts.one_launch
    g_all = _games(every.drain_replay())
    q = np.concatenate([x[4] for x in g_all.values()])
    v = float(np.float32(np.quantile(q, 0.05)))
    on = _run(512, 16, 90, evaluator=mcts.FusedNetEvaluator(model), resign_threshold=v, resign_audit=0.0, **kw)
    assert _check_prefixes(_games(on.drain_replay()), g_all, v, min_common=256) > 16


def test_off_means_off():
    """resign_threshold=None launches what self-play launches without the option and gives the same records, no q"""
    kw = dict(size=4, temp_plies=20, seed=9)
    a = _run(32, 8, 30, **kw)
    b = _run(32, 8, 30, resign_threshold=None, resign_audit=0.5, **kw)
    assert b.rs is None and b.resign_threshold is None and a.total_launches() == b.total_launches()
    sa, sb = a.stats(), b.stats()
    assert sa == sb and sb["resigned"] == sb["audited"] == 0
    ra, rb = a.drain_replay(), b.drain_replay()
    assert "q" not in rb and sorted(ra) == sorted(rb)
    ga, gb = _games(ra), _games(rb)  # rows are in reservation order, which the warps' timing decides
    assert sorted(ga) == sorted(gb) and all(_same(ga[g], gb[g]) for g in ga)
    with pytest.raises(RuntimeError, match="set_resign_threshold"):
        b.set_resign_threshold(0.0)


def test_threshold_changes_between_plies():
    """-1 for the first plies (nothing resigns), then 1.0: every game that is not audited resigns at its next ply"""
    sp = _run(64, 8, 6, size=6, temp_plies=10, seed=2, resign_threshold=-1.0, resign_audit=0.0)
    assert sp.stats()["resigned"] == 0 and sp.resign_threshold == -1.0
    sp.set_resign_threshold(1.0)
    sp.play_move()
    st = sp.stats()
    assert st["resigned"] == 64 and st["games"] == 64 and sp.ply.tolist() == [0] * 64
    got = _games(sp.drain_replay())
    assert all(len(x[0]) == 7 and x[3][-1] == -1 for x in got.values())


def C_offset(t, k):
    import ctypes

    return ctypes.c_void_p(t.data_ptr() + k)


def test_refusals():
    from betazero_b200 import _lib, mcts, selfplay

    L = _lib.load()
    for empties in (0, 10):
        sp = selfplay.BatchedSelfPlay(8, 8, mcts.HashEvaluator(1), board_size=6, endgame_empties=empties, use_graph=False,
                                      resign_threshold=0.0)
        sp.search()
        rs, eg = sp.rs, (sp._eg_ref if sp.eg is not None else None)

        def advance():
            return L.bz_selfplay_advance_resign(sp._ref, eg, sp._rs_ref, sp.pools._ref, None, _lib.stream_ptr())

        def play():
            return L.bz_selfplay_endgame_play_resign(sp._ref, eg, sp._rs_ref, _lib.dptr(sp.eg_workspace), 0,
                                                     _lib.stream_ptr())

        bad = [("threshold", float("nan")), ("threshold", 1.5), ("threshold", -1.01), ("audit_below", (1 << 32) + 1),
               ("hist_q", None), ("rp_q", None), ("counters", None)]
        if empties:
            bad.append(("eg_hist_q", None))
        for field, value in bad:
            old = getattr(rs, field)
            setattr(rs, field, value)
            assert advance() == -1, field
            if empties:
                assert play() == -1, field
            setattr(rs, field, old)
        assert L.bz_selfplay_advance_resign(sp._ref, eg, None, sp.pools._ref, None, _lib.stream_ptr()) == -1
        rs.audit_below = 1 << 32  # every game audited: accepted
        assert advance() == 0
        if empties:
            assert L.bz_selfplay_endgame_play_resign(sp._ref, eg, None, _lib.dptr(sp.eg_workspace), 0,
                                                     _lib.stream_ptr()) == -1
            assert L.bz_selfplay_endgame_play_resign(sp._ref, eg, sp._rs_ref, C_offset(sp.eg_workspace, 4), 0,
                                                     _lib.stream_ptr()) == -2
            assert play() == 0
        else:
            assert L.bz_selfplay_endgame_play_resign(sp._ref, None, sp._rs_ref, None, 0, _lib.stream_ptr()) == -1
        torch.cuda.synchronize()
        sp.mcts.check_errors()


def test_loop_calibrates_and_resumes_the_threshold(tmp_path):
    import math

    from betazero_b200 import loop

    ck = str(tmp_path / "ck.pt")
    args = loop.default_args(games=256, sims=16, leaves=4, plies=70, train_steps=2, batch=256, lr=1e-3, iterations=2,
                             resign_fp=0.05, resign_audit=0.5, checkpoint=ck)
    l1, l2 = loop.run(args)
    r1, r2 = l1["resign"], l2["resign"]
    assert r1["threshold"] == -1.0 and r1["resigned_local"] == 0 and r1["audited_games"] > 0 and r1["fp"] == 0.0
    assert -1.0 <= r1["next_threshold"] <= 1.0 and r2["threshold"] == r1["next_threshold"]
    assert r1["audited_local"] > 0 and r1["plies_per_game"] > 0 and r2["fp_target"] == 0.05
    assert all(math.isfinite(x) for x in l2["loss_first_last"])
    resumed = loop.default_args(games=256, sims=16, leaves=4, plies=4, train_steps=1, batch=256, resume=ck, resign=-1.0)
    (l3,) = loop.run(resumed)
    assert l3["resign"]["threshold"] == r2["next_threshold"] and l3["resign"]["next_threshold"] == r2["next_threshold"]
    fixed = loop.default_args(games=48, sims=16, plies=2, size=6, train_steps=1, batch=64)
    assert "resign" not in loop.run_iteration(loop.LoopState(fixed, 0, 1), 0)
