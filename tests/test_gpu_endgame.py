"""The endgame solver on the GPU: bz_endgame_solve equals the C oracle's plain negamax (oracle/endgame.c
orc_endgame_solve) bit for bit in action, value and every move value, visits at most its nodes, and is consistent with
itself where the oracle is too slow; PerfectPlayer plays perfect 4x4 games; the endgame suite and its metrics
(betazero_b200/endgame.py); loop.py --eval-endgame."""
import ctypes

import numpy as np
import pytest
import torch

from helpers import _minimax_bounds_checks  # noqa: F401

pytestmark = pytest.mark.gpu


def _dev(x):
    from betazero_b200 import env

    return env.to_device_u64(np.ascontiguousarray(x, np.uint64))


def _late_positions(size, n, max_empties, seed):
    """mover-relative positions from random games with 0 .. max_empties empties, spread evenly over the counts: roots
    that must pass and finished games included"""
    from oracle import pyoracle as po

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


def _gpu(me, opp, size):
    from betazero_b200 import minimax

    a, v, mv, n = minimax.solve(_dev(me), _dev(opp), size)
    return a.cpu().numpy(), v.cpu().numpy(), mv.cpu().numpy(), n.cpu().numpy()


@pytest.mark.parametrize("size,n,max_empties", [(8, 2200, 10), (6, 390, 12), (4, 260, 12)])
def test_solve_equals_the_c_oracle(size, n, max_empties):
    from oracle import pyendgame as pe

    me, opp = _late_positions(size, n, max_empties, seed=size)
    if size == 4:  # the start position: the whole game
        me, opp = np.append(me, np.uint64(0x40200)), np.append(opp, np.uint64(0x20400))
    a, v, mv, nodes = _gpu(me, opp, size)
    ra, rv, rmv, rn = pe.endgame_solve(me, opp, size)
    assert np.array_equal(a, ra) and np.array_equal(v, rv) and np.array_equal(mv, rmv)
    assert (nodes >= 1).all() and (nodes <= rn).all()  # alpha-beta enters at most what plain negamax enters
    e = _empties(me, opp, size)
    assert set(e.tolist()) >= set(range(1, max_empties + 1))
    big = e >= 8
    assert nodes[big].sum() < rn[big].sum()  # the pruning prunes
    assert (a == 64).any() and (a == 255).any()
    if size == 4:
        assert v[-1] == -8 and a[-1] == 2


def test_solve_equals_the_c_oracle_at_12_empties():
    from betazero_b200 import endgame
    from oracle import pyendgame as pe

    s = endgame.positions(8, 12, 8, seed=3)
    me, opp = s.me.cpu().numpy().view(np.uint64), s.opp.cpu().numpy().view(np.uint64)
    a, v, mv, nodes = _gpu(me, opp, 8)
    ra, rv, rmv, rn = pe.endgame_solve(me, opp, 8)
    assert np.array_equal(a, ra) and np.array_equal(v, rv) and np.array_equal(mv, rmv) and (nodes <= rn).all()
    assert nodes.sum() < rn.sum()


def test_a_result_does_not_depend_on_the_batch():
    me, opp = _late_positions(8, 600, 10, seed=21)
    a, v, mv, n = _gpu(me, opp, 8)
    perm = np.random.default_rng(0).permutation(600)
    pme, popp = _late_positions(8, 300, 9, seed=22)
    a2, v2, mv2, n2 = _gpu(np.concatenate([me[perm], pme]), np.concatenate([opp[perm], popp]), 8)
    assert np.array_equal(a2[:600], a[perm]) and np.array_equal(v2[:600], v[perm])
    assert np.array_equal(mv2[:600], mv[perm]) and np.array_equal(n2[:600], n[perm])
    for i in range(0, 600, 97):  # alone
        a1, v1, mv1, n1 = _gpu(me[i:i + 1], opp[i:i + 1], 8)
        assert (a1[0], v1[0], n1[0]) == (a[i], v[i], n[i]) and np.array_equal(mv1[0], mv[i])


@pytest.mark.parametrize("size,empties,n", [(8, 14, 12), (6, 16, 8)])
def test_move_values_are_the_childrens_values(size, empties, n):
    """beyond the oracle's reach: every move's value is minus its child's value solved as a root, and the value is
    their maximum (16 empties on 6x6: one 8x8 root with 14 empties already took 651 M nodes)"""
    from betazero_b200 import endgame, env, minimax

    s = endgame.positions(n, empties, size, seed=empties)
    a, v, mv, _ = minimax.solve(s.me, s.opp, size)
    a, v, mv = a.cpu().numpy(), v.cpu().numpy(), mv.cpu().numpy().astype(np.int64)
    rows, acts = np.nonzero(mv[:, :64] != -128)
    cme, copp, _ = env.apply(s.me[torch.from_numpy(rows).cuda()], s.opp[torch.from_numpy(rows).cuda()],
                             torch.from_numpy(acts.astype(np.uint8)).cuda(), size)
    _, cv, _, _ = minimax.solve(cme, copp, size)
    assert np.array_equal(mv[rows, acts], -cv.cpu().numpy().astype(np.int64))
    for i in range(n):
        legal = mv[i] != -128
        assert v[i] == mv[i][legal].max() and a[i] == int(np.argmax(np.where(legal, mv[i], -200)))


def test_refusals():
    from betazero_b200 import _lib, minimax, players
    from betazero_b200.boards import ReversiBoard

    L, st = _lib.load(), _lib.stream_ptr()
    me, opp = _dev([0x0000000810000000]), _dev([0x0000001008000000])  # the 8x8 start: 60 empties
    with pytest.raises(ValueError):
        minimax.solve(me, opp, 8)
    with pytest.raises(ValueError):
        players.PerfectPlayer(1, 8).get_move(ReversiBoard(size=8))
    with pytest.raises(ValueError):
        minimax.solve(me, opp, 5)
    a, v = torch.empty(1, dtype=torch.uint8, device="cuda"), torch.empty(1, dtype=torch.int8, device="cuda")
    mv, n = torch.empty(65, dtype=torch.int8, device="cuda"), torch.empty(1, dtype=torch.int64, device="cuda")
    ws = torch.empty(int(L.bz_endgame_workspace_bytes(1)) + 16, dtype=torch.uint8, device="cuda")
    ins, outs = [_lib.dptr(me), _lib.dptr(opp)], [_lib.dptr(a), _lib.dptr(v), _lib.dptr(mv), _lib.dptr(n)]
    for bad_size in (0, 5, 7, 10):
        assert L.bz_endgame_solve(*ins, 1, bad_size, _lib.dptr(ws), *outs, st) == -1
    assert L.bz_endgame_solve(*ins, -1, 8, _lib.dptr(ws), *outs, st) == -1
    assert L.bz_endgame_solve(*ins, 1 << 25, 8, _lib.dptr(ws), *outs, st) == -1
    assert L.bz_endgame_solve(None, ins[1], 1, 8, _lib.dptr(ws), *outs, st) == -1
    assert L.bz_endgame_solve(*ins, 1, 8, None, *outs, st) == -1
    for k in range(3):
        bad = list(outs)
        bad[k] = None
        assert L.bz_endgame_solve(*ins, 1, 8, _lib.dptr(ws), *bad, st) == -1
    assert L.bz_endgame_solve(*ins, 1, 8, ctypes.c_void_p(ws.data_ptr() + 8), *outs, st) == -2
    assert L.bz_endgame_solve(*ins, 0, 8, None, None, None, None, None, st) == 0  # nothing to do
    # the kernel itself does not search a root with too many empties
    assert L.bz_endgame_solve(*ins, 1, 8, _lib.dptr(ws), *outs[:3], None, st) == 0
    torch.cuda.synchronize()
    assert (int(a[0]), int(v[0])) == (255, 0) and (mv.cpu().numpy() == -128).all()
    assert L.bz_endgame_solve(*ins, 1, 8, _lib.dptr(ws), *outs, st) == 0
    torch.cuda.synchronize()
    assert int(n[0]) == 0
    if hasattr(L, "bz_debug_checks_minimax"):  # the bounds-check build records the refused root; clear the record
        rec = (ctypes.c_int * 4)()
        assert L.bz_debug_checks_minimax(rec) == 0 and rec[0] == 70


def _score_x(winner_counts):
    _, (c1, c2), _ = winner_counts
    return c1 - c2


def test_perfect_players_on_4x4():
    from betazero_b200 import arena, players
    from betazero_b200.boards import ReversiBoard

    assert _score_x(arena.play_game(ReversiBoard, players.PerfectPlayer(1, 4), players.PerfectPlayer(-1, 4), size=4)) == -8
    for seed in range(4):
        for opp_of in (lambda s: players.RandomPlayer(s, size=4, seed=seed), lambda s: players.OptimalPlayer(s, 2, size=4)):
            assert _score_x(arena.play_game(ReversiBoard, players.PerfectPlayer(1, 4), opp_of(-1), size=4)) >= -8
            assert _score_x(arena.play_game(ReversiBoard, opp_of(1), players.PerfectPlayer(-1, 4), size=4)) <= -8


def test_suite_is_fixed_by_its_seed():
    from betazero_b200 import endgame, env

    for size, e in ((8, 12), (6, 8)):
        s1, s2 = endgame.positions(300, e, size, seed=5), endgame.positions(300, e, size, seed=5)
        assert torch.equal(s1.me, s2.me) and torch.equal(s1.opp, s2.opp)
        s3 = endgame.positions(300, e, size, seed=6)
        assert not torch.equal(s1.me, s3.me)
        me, opp = env.to_host_u64(s1.me), env.to_host_u64(s1.opp)
        assert (_empties(me, opp, size) == e).all()
        moves = np.array([bin(int(x)).count("1") for x in env.to_host_u64(env.legal_mask(s1.me, s1.opp, size))])
        assert (moves >= 2).all()
        assert len({(int(a), int(b)) for a, b in zip(me, opp)}) > 250  # mostly distinct positions


def test_evaluate_plays_the_players_moves_and_scores_them():
    from betazero_b200 import endgame, minimax, net, players
    from betazero_b200.boards import ReversiBoard
    from oracle import pyoracle as po

    suite = endgame.solve_suite(endgame.positions(256, 10, 8, seed=1))
    me, opp = endgame.env.to_host_u64(suite.me), endgame.env.to_host_u64(suite.opp)

    def board(i):
        b = ReversiBoard(size=8)
        b.board = po.wire_to_grid(me[i], opp[i], 8, 1)
        return b

    # budget 0: the raw policy is GreedyNetPlayer's move
    fnet = net.make_net("mlp", seed=4, dtype=torch.float32)
    played, head = endgame.raw_policy(fnet, suite.me, suite.opp, 8)
    g = players.GreedyNetPlayer(1, fnet, size=8)
    for i in range(0, 256, 16):
        r, c = g.get_move(board(i))
        assert played[i] == r * 8 + c, i
    # a budget: the one-launch search's move is MCTSPlayer's
    model = net.make_net("mlp", seed=2)
    moves = endgame.searched_moves(model, suite.me, suite.opp, 64, n_leaves=4, size=8)
    for i in range(0, 256, 32):
        r, c = players.MCTSPlayer(1, net=model, n_sims=64, size=8, n_leaves=4).get_move(board(i))
        assert moves[i] == r * 8 + c, i
    # the metrics, recomputed from the move values
    r = endgame.evaluate(model, suite, sims=(0, 64), n_leaves=4, minimax_depths=(2,))
    mv, best = suite.move_value.astype(np.int64), suite.value.astype(np.int64)
    for s, pl in (("64", moves), ("0", endgame.raw_policy(model, suite.me, suite.opp, 8)[0])):
        pv = mv[np.arange(256), pl]
        assert r["budgets"][s]["move_accuracy"] == pytest.approx(np.mean(pv == best))
        assert r["budgets"][s]["wld_accuracy"] == pytest.approx(np.mean(np.sign(pv) == np.sign(best)))
        assert r["budgets"][s]["mean_disc_loss"] == pytest.approx(np.mean(best - pv))
    assert "value_mse" in r["budgets"]["0"] and "value_mse" not in r["budgets"]["64"]
    ma, _, _ = minimax.best_moves(suite.me, suite.opp, 2, 8, seed=suite.seed,
                                  keys=torch.arange(256, dtype=torch.int64, device="cuda"))
    pv = mv[np.arange(256), ma.long().cpu().numpy()]
    assert r["baselines"]["minimax2"]["move_accuracy"] == pytest.approx(np.mean(pv == best))
    n_opt = (mv == best[:, None]).sum(1)
    assert r["baselines"]["random"]["move_accuracy"] == pytest.approx(np.mean(n_opt / (mv != -128).sum(1)))


def test_loop_reports_eval_endgame(monkeypatch):
    from betazero_b200 import loop, minimax

    calls = []
    solve = minimax.solve
    monkeypatch.setattr(minimax, "solve", lambda *a, **k: calls.append(1) or solve(*a, **k))
    args = loop.default_args(games=48, sims=16, leaves=4, plies=6, size=6, train_steps=2, batch=128, lr=1e-2,
                             iterations=2, eval_endgame=8)
    lines = loop.run(args)
    assert len(calls) == 1
    for ln in lines:
        e = ln["eval_endgame"]
        assert e["empties"] == 8 and e["positions"] == loop.ENDGAME_POSITIONS and set(e["budgets"]) == {"0", "16"}
        assert 0.0 <= e["budgets"]["16"]["move_accuracy"] <= 1.0
    assert "eval_endgame" not in loop.run_iteration(loop.LoopState(loop.default_args(games=48, sims=16, plies=2, size=6,
                                                                                     train_steps=1, batch=64), 0, 1), 0)
    with pytest.raises(ValueError):
        loop.LoopState(loop.default_args(games=48, sims=16, size=6, eval_endgame=21), 0, 1)
