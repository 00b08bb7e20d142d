"""The win/draw/loss solver on the GPU: bz_endgame_solve_wld equals the sign transform of the C oracle's plain negamax
(oracle/endgame_wld_ref.py endgame_solve_wld) bit for bit in action, value and every move value and enters at most its
nodes;
it agrees in sign with the exact solver on the seed-0 suites with fewer nodes; it is consistent with itself beyond the
exact solver's reach; its results do not depend on the batch; its refusals.  The WLD handover
(BatchedSelfPlay(endgame_solve="wld"); bz_selfplay_endgame_play_wld) against the sequential restatement
(oracle/selfplay_endgame_ref.py with endgame_wld_ref.wld_solver) and against the exact handover; endgame.evaluate on a
WLD suite; loop.py --endgame-solve wld."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import endgame_wld_ref as ewr
from oracle import mcts_ref as mr
from oracle import pyoracle as po
from oracle import selfplay_endgame_ref as ser

from helpers import _minimax_bounds_checks  # noqa: F401

pytestmark = pytest.mark.gpu


def _dev(x):
    from betazero_b200 import env

    return env.to_device_u64(np.ascontiguousarray(x, np.uint64))


def _late_positions(size, n, max_empties, seed):
    """mover-relative positions from random games with 0 .. max_empties empties, spread evenly over the counts: roots
    that must pass and finished games included"""
    rng = np.random.default_rng(seed)
    per = -(-n // (max_empties + 1))
    me, opp, have = [], [], {e: 0 for e in range(max_empties + 1)}
    k = 0
    while len(me) < n:
        e_want = int(rng.integers(0, max_empties + 1))
        g, pl, _, _ = po.random_playout(size, seed * 100_003 + k, size * size - 4 - e_want + int(rng.integers(0, 2)))
        k += 1
        m, o = po.grid_to_wire(g, pl)
        e = size * size - bin(m | o).count("1")
        if e <= max_empties and have[e] < per:
            have[e] += 1
            me.append(m)
            opp.append(o)
    return np.array(me, np.uint64), np.array(opp, np.uint64)


def _empties(me, opp, size):
    return size * size - np.array([bin(int(a) | int(b)).count("1") for a, b in zip(me, opp)])


def _wld(me, opp, size):
    from betazero_b200 import minimax

    a, v, mv, n = minimax.solve(_dev(me), _dev(opp), size, wld=True)
    return a.cpu().numpy(), v.cpu().numpy(), mv.cpu().numpy(), n.cpu().numpy()


def _host(t):
    return t.cpu().numpy().view(np.uint64)


@pytest.mark.parametrize("size,n,max_empties", [(8, 2200, 10), (6, 390, 12), (4, 260, 12)])
def test_solve_wld_equals_the_sign_transformed_c_oracle(size, n, max_empties):
    me, opp = _late_positions(size, n, max_empties, seed=40 + size)
    if size == 4:  # the start position: the whole game, a loss for the first player
        me, opp = np.append(me, np.uint64(0x40200)), np.append(opp, np.uint64(0x20400))
    a, v, mv, nodes = _wld(me, opp, size)
    ra, rv, rmv, rn = ewr.endgame_solve_wld(me, opp, size)
    assert np.array_equal(a, ra) and np.array_equal(v, rv) and np.array_equal(mv, rmv)
    assert (nodes >= 1).all() and (nodes <= rn).all()  # alpha-beta enters at most what plain negamax enters
    e = _empties(me, opp, size)
    assert set(e.tolist()) >= set(range(1, max_empties + 1))
    assert (a == 64).any() and (a == 255).any() and {-1, 1} <= set(v.tolist()) <= {-1, 0, 1}
    if size == 4:
        assert v[-1] == -1 and a[-1] == 2


def test_solve_wld_equals_the_sign_transformed_c_oracle_at_12_empties():
    from betazero_b200 import endgame

    s = endgame.positions(8, 12, 8, seed=3)
    me, opp = _host(s.me), _host(s.opp)
    a, v, mv, nodes = _wld(me, opp, 8)
    ra, rv, rmv, rn = ewr.endgame_solve_wld(me, opp, 8)
    assert np.array_equal(a, ra) and np.array_equal(v, rv) and np.array_equal(mv, rmv) and (nodes <= rn).all()


@pytest.mark.parametrize("empties,n", [(12, 4096), (14, 32)])
def test_agrees_in_sign_with_the_exact_solver_on_the_suites(empties, n):
    """the seed-0 suites of the probes: every value and move value is the sign of the exact one; at 12 empties the WLD
    search enters fewer nodes in total (a deterministic count, not a timing)"""
    from betazero_b200 import endgame, minimax

    s = endgame.positions(n, empties, 8, seed=0)
    _, v, mv, nodes = minimax.solve(s.me, s.opp, 8)
    a_w, v_w, mv_w, nodes_w = minimax.solve(s.me, s.opp, 8, wld=True)
    v, mv, v_w, mv_w = v.cpu().numpy(), mv.cpu().numpy(), v_w.cpu().numpy(), mv_w.cpu().numpy()
    assert np.array_equal(v_w, np.sign(v)) and np.array_equal(mv_w, np.where(mv == -128, mv, np.sign(mv)))
    a_w = a_w.long().cpu().numpy()
    assert (mv_w[np.arange(n), a_w] == v_w).all()
    if empties == 12:
        assert int(nodes_w.sum()) < int(nodes.sum())


@pytest.mark.parametrize("size,empties,n", [(8, 16, 16), (6, 18, 12)])
def test_move_values_are_the_childrens_results(size, empties, n):
    """beyond the exact solver's reach: every move's result is minus its child's result solved as a root, and the
    root's is their maximum, with the action the first move that keeps it"""
    from betazero_b200 import endgame, env, minimax

    s = endgame.positions(n, empties, size, seed=empties)
    a, v, mv, _ = minimax.solve(s.me, s.opp, size, wld=True)
    a, v, mv = a.cpu().numpy(), v.cpu().numpy(), mv.cpu().numpy().astype(np.int64)
    rows, acts = np.nonzero(mv[:, :64] != -128)
    cme, copp, _ = env.apply(s.me[torch.from_numpy(rows).cuda()], s.opp[torch.from_numpy(rows).cuda()],
                             torch.from_numpy(acts.astype(np.uint8)).cuda(), size)
    _, cv, _, _ = minimax.solve(cme, copp, size, wld=True)
    assert np.array_equal(mv[rows, acts], -cv.cpu().numpy().astype(np.int64))
    for i in range(n):
        legal = mv[i] != -128
        assert v[i] == mv[i][legal].max() and a[i] == int(np.argmax(np.where(legal, mv[i], -200)))


def test_a_result_does_not_depend_on_the_batch():
    me, opp = _late_positions(8, 600, 10, seed=61)
    a, v, mv, n = _wld(me, opp, 8)
    perm = np.random.default_rng(0).permutation(600)
    pme, popp = _late_positions(8, 300, 9, seed=62)
    a2, v2, mv2, n2 = _wld(np.concatenate([me[perm], pme]), np.concatenate([opp[perm], popp]), 8)
    assert np.array_equal(a2[:600], a[perm]) and np.array_equal(v2[:600], v[perm])
    assert np.array_equal(mv2[:600], mv[perm]) and np.array_equal(n2[:600], n[perm])
    for i in range(0, 600, 97):  # alone
        a1, v1, mv1, n1 = _wld(me[i:i + 1], opp[i:i + 1], 8)
        assert (a1[0], v1[0], n1[0]) == (a[i], v[i], n[i]) and np.array_equal(mv1[0], mv[i])


def test_refusals():
    from betazero_b200 import _lib, minimax

    L, st = _lib.load(), _lib.stream_ptr()
    me, opp = _dev([0x0000000810000000]), _dev([0x0000001008000000])  # the 8x8 start: 60 empties
    with pytest.raises(ValueError):
        minimax.solve(me, opp, 8, wld=True)
    with pytest.raises(ValueError):
        minimax.solve(me, opp, 5, wld=True)
    a, v = torch.empty(1, dtype=torch.uint8, device="cuda"), torch.empty(1, dtype=torch.int8, device="cuda")
    mv, n = torch.empty(65, dtype=torch.int8, device="cuda"), torch.empty(1, dtype=torch.int64, device="cuda")
    ws = torch.empty(int(L.bz_endgame_workspace_bytes(1)) + 16, dtype=torch.uint8, device="cuda")
    ins, outs = [_lib.dptr(me), _lib.dptr(opp)], [_lib.dptr(a), _lib.dptr(v), _lib.dptr(mv), _lib.dptr(n)]
    for bad_size in (0, 5, 7, 10):
        assert L.bz_endgame_solve_wld(*ins, 1, bad_size, _lib.dptr(ws), *outs, st) == -1
    assert L.bz_endgame_solve_wld(*ins, -1, 8, _lib.dptr(ws), *outs, st) == -1
    assert L.bz_endgame_solve_wld(*ins, 1 << 25, 8, _lib.dptr(ws), *outs, st) == -1
    assert L.bz_endgame_solve_wld(None, ins[1], 1, 8, _lib.dptr(ws), *outs, st) == -1
    assert L.bz_endgame_solve_wld(*ins, 1, 8, None, *outs, st) == -1
    for k in range(3):
        bad = list(outs)
        bad[k] = None
        assert L.bz_endgame_solve_wld(*ins, 1, 8, _lib.dptr(ws), *bad, st) == -1
    assert L.bz_endgame_solve_wld(*ins, 1, 8, ctypes.c_void_p(ws.data_ptr() + 8), *outs, st) == -2
    assert L.bz_endgame_solve_wld(*ins, 0, 8, None, None, None, None, None, st) == 0  # nothing to do
    # the kernel itself does not search a root with too many empties
    assert L.bz_endgame_solve_wld(*ins, 1, 8, _lib.dptr(ws), *outs[:3], None, st) == 0
    torch.cuda.synchronize()
    assert (int(a[0]), int(v[0])) == (255, 0) and (mv.cpu().numpy() == -128).all()
    assert L.bz_endgame_solve_wld(*ins, 1, 8, _lib.dptr(ws), *outs, st) == 0
    torch.cuda.synchronize()
    assert int(n[0]) == 0
    if hasattr(L, "bz_debug_checks_minimax"):  # the bounds-check build records the refused root; clear the record
        rec = (ctypes.c_int * 4)()
        assert L.bz_debug_checks_minimax(rec) == 0 and rec[0] == 70


# ---- the WLD handover ------------------------------------------------------------------------------------------------

def _games(rp):
    """game id -> (me, opp, pi, z) in ply order; every game's plies are 0 .. n-1"""
    game, ply = rp["game"].cpu().numpy(), rp["ply"].cpu().numpy()
    me, opp = rp["me"].cpu().numpy().view(np.uint64), rp["opp"].cpu().numpy().view(np.uint64)
    pi, z = rp["pi"].cpu().numpy(), rp["z"].cpu().numpy()
    out = {}
    order = np.lexsort((ply, game))
    for idx in np.split(order, np.flatnonzero(np.diff(game[order])) + 1):
        if idx.size:
            assert np.array_equal(ply[idx], np.arange(idx.size))
            out[int(game[idx[0]])] = (me[idx], opp[idx], pi[idx], z[idx])
    return out


@pytest.mark.parametrize("size,n_sims,empties,leaves", [(4, 24, 6, 1), (4, 24, 6, 4), (6, 16, 10, 1), (6, 16, 10, 4),
                                                       (8, 32, 8, 1), (8, 32, 8, 4), (8, 32, 12, 1), (8, 32, 12, 4)])
def test_deterministic_wld_handover_equals_sequential_restatement(size, n_sims, empties, leaves):
    """temp_plies = 0: every slot plays the restatement's game; actions, records, z, counters, restarts and game ids"""
    from betazero_b200 import mcts, selfplay

    salt = 3
    game = mr.ReversiGame(po.OracleReversiBoard, size)
    hist, winner, h = ser.self_play_game_endgame(game, n_sims, 1.25, lambda a, b: mr.hash_eval(a, b, salt, 65), empties,
                                                 solve=ewr.wld_solver(ser.c_solver(game)), leaves=leaves)
    assert h is not None
    B = 5
    sp = selfplay.BatchedSelfPlay(B, n_sims, mcts.HashEvaluator(salt), board_size=size, temp_plies=0, use_graph=False,
                                  rank=1, world=3, n_leaves=leaves, endgame_empties=empties, endgame_every=1,
                                  endgame_solve="wld")
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

    sp = selfplay.BatchedSelfPlay(B, n_sims, mcts.HashEvaluator(7), board_size=size, use_graph=False, **kw)
    for _ in range(plies):
        sp.play_move()
    sp.mcts.check_errors()
    return sp


def test_wld_handover_keeps_the_prefix_and_z_of_the_exact_handover():
    """sampled moves, the same seed: every record before a game's handover is the exact handover's, every z is, and at
    the handover position the WLD pi's support contains the exact pi's (an exact-optimal move keeps the result)"""
    E = 8
    kw = dict(temp_plies=24, seed=11, endgame_empties=E)
    ex = _run(128, 16, 140, **kw)
    wl = _run(128, 16, 140, endgame_solve="wld", **kw)
    for sp in (ex, wl):
        st = sp.stats()
        assert st["endgame_overflow"] == 0 and st["endgame_games"] > 128 and st["dropped"] == 0
    assert ex.game_id.tolist() == wl.game_id.tolist()  # the slots restart at the same plies
    ge, gw = _games(ex.drain_replay()), _games(wl.drain_replay())
    common = sorted(set(ge) & set(gw))
    assert len(common) >= 128
    handed = wider = 0
    for g in common:
        me, opp, pi, z = gw[g]
        eme, eopp, epi, ez = ge[g]
        e = _empties(me, opp, 8)
        h = int(np.argmax(e <= E)) if (e <= E).any() else len(me)
        assert np.array_equal(me[:h + 1], eme[:h + 1]) and np.array_equal(opp[:h + 1], eopp[:h + 1]), g
        assert np.array_equal(pi[:h], epi[:h]), g
        if h == len(me):
            assert len(eme) == h and np.array_equal(z, ez), g
            continue
        handed += 1
        assert np.array_equal(z[:h + 1], ez[:h + 1]), g  # the same outcome
        sign = np.where(np.arange(len(me)) % 2 == h % 2, 1, -1)
        assert np.array_equal(z, z[h] * sign), g
        assert ((epi[h] > 0) <= (pi[h] > 0)).all(), g
        wider += int((pi[h] > 0).sum() > (epi[h] > 0).sum())
    assert handed >= 64 and wider > 0


def test_evaluate_on_a_wld_suite():
    """the same positions as an exact and as a WLD suite: equal wld_accuracy for every budget and baseline, equal value
    metrics, and no move_accuracy / mean_disc_loss on the WLD side"""
    from betazero_b200 import endgame, net

    exact = endgame.positions(512, 10, 8, seed=1)
    wld = endgame.Suite(exact.me, exact.opp, exact.size, exact.empties, exact.seed, wld=True)
    model = net.make_net("mlp", seed=2)
    re = endgame.evaluate(model, exact, sims=(0, 64), n_leaves=4, minimax_depths=(2,))
    rw = endgame.evaluate(model, wld, sims=(0, 64), n_leaves=4, minimax_depths=(2,))
    assert set(np.unique(wld.value).tolist()) <= {-1, 0, 1} and np.array_equal(wld.value, np.sign(exact.value))
    for s in ("0", "64"):
        assert rw["budgets"][s]["wld_accuracy"] == re["budgets"][s]["wld_accuracy"]
        assert "move_accuracy" not in rw["budgets"][s] and "mean_disc_loss" not in rw["budgets"][s]
    for k in ("value_sign_accuracy", "value_mse"):
        assert rw["budgets"]["0"][k] == re["budgets"]["0"][k]
    for b in ("random", "minimax2"):
        assert rw["baselines"][b] == {"wld_accuracy": re["baselines"][b]["wld_accuracy"]}
    assert endgame.solve_stats(wld)["solve"] == "wld" and endgame.solve_stats(exact)["solve"] == "exact"
    assert endgame.solve_stats(wld)["nodes"] < endgame.solve_stats(exact)["nodes"]


def test_loop_with_the_wld_solver():
    from betazero_b200 import loop

    def lines(solve):
        return loop.run(loop.default_args(games=48, sims=16, leaves=4, plies=28, size=6, train_steps=2, batch=128,
                                          lr=1e-2, iterations=2, endgame_empties=10, endgame_every=4, eval_endgame=8,
                                          endgame_solve=solve))

    wl, ex = lines("wld"), lines("exact")
    for lw, le in zip(wl, ex):
        assert lw["endgame"]["solve"] == "wld" and le["endgame"]["solve"] == "exact"
        assert lw["eval_endgame"]["solve"] == "wld" and le["eval_endgame"]["solve"] == "exact"
        assert set(lw["endgame"]) == set(le["endgame"]) and lw["endgame"]["games"] > 0 and lw["endgame"]["ms"] > 0
        assert set(lw["eval_endgame"]) == set(le["eval_endgame"]) and set(lw["eval_endgame"]["budgets"]) == {"0", "16"}
        assert set(lw["eval_endgame"]["budgets"]["16"]) == {"wld_accuracy"}
        assert lw["eval_endgame"]["random"] == {"wld_accuracy": le["eval_endgame"]["random"]["wld_accuracy"]}
    # the first iteration's self-play (the same net) hands the same games over at the same plies
    assert wl[0]["endgame"]["games"] == ex[0]["endgame"]["games"]
    assert wl[0]["games_finished_local"] == ex[0]["games_finished_local"]
