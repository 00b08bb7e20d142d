"""Minimax players on the GPU: bz_minimax_moves equals the C oracle's plain minimax (oracle/minimax.c) bit for bit, move
and value; OptimalPlayer / RandomPlayer equal the definition (oracle/minimax_ref.py) move for move; tournaments with
minimax entrants play the games the sequential players play."""
import ctypes

import numpy as np
import pytest
import torch

from helpers import _minimax_bounds_checks  # noqa: F401

pytestmark = pytest.mark.gpu


def _dev(x):
    from betazero_b200 import env

    return env.to_device_u64(np.ascontiguousarray(x, np.uint64))


def _set(size, n, max_depth, seed):
    """positions of every stage (random playouts: passes and finished games included), a depth and a key each"""
    from oracle import pyoracle as po

    me, opp = po.playout_boards(n, seed=seed, size=size)
    rng = np.random.default_rng(seed)
    return me, opp, rng.integers(0, max_depth + 1, n).astype(np.uint8), rng.integers(0, 2**32, n).astype(np.uint64)


def _gpu(me, opp, depth, keys, seed, size):
    from betazero_b200 import minimax

    a, v, n = minimax.best_moves(_dev(me), _dev(opp), torch.from_numpy(depth.astype(np.int64)),
                                 size=size, seed=seed, keys=torch.from_numpy(keys.astype(np.int64)))
    return a.cpu().numpy(), v.cpu().numpy(), n.cpu().numpy()


@pytest.mark.parametrize("size,n,max_depth", [(8, 2048, 5), (6, 1536, 7), (4, 1024, 8)])
def test_moves_equal_the_c_oracle(size, n, max_depth):
    from oracle import pyminimax as pm

    me, opp, depth, keys = _set(size, n, max_depth, seed=size)
    a, v, nodes = _gpu(me, opp, depth, keys, 17, size)
    ra, rv, rn = pm.minimax_moves(me, opp, depth, keys, seed=17, size=size)
    assert np.array_equal(a, ra) and np.array_equal(v, rv)
    assert (nodes >= 1).all() and (nodes <= rn).all()  # alpha-beta visits at most what plain minimax visits
    assert (a == 64).any() and (a == 255).any() and (np.abs(v) == 127).any() and set(depth.tolist()) == set(range(max_depth + 1))
    if size == 8:
        assert nodes[depth == 5].sum() < rn[depth == 5].sum()  # the pruning prunes


def test_a_result_does_not_depend_on_the_batch():
    me, opp, depth, keys = _set(8, 700, 4, seed=21)
    a, v, n = _gpu(me, opp, depth, keys, 3, 8)
    perm = np.random.default_rng(0).permutation(700)
    pad_me, pad_opp, pad_d, pad_k = _set(8, 300, 6, seed=22)
    bme = np.concatenate([me[perm], pad_me])
    bopp = np.concatenate([opp[perm], pad_opp])
    bd = np.concatenate([depth[perm], pad_d])
    bk = np.concatenate([keys[perm], pad_k])
    a2, v2, n2 = _gpu(bme, bopp, bd, bk, 3, 8)
    assert np.array_equal(a2[:700], a[perm]) and np.array_equal(v2[:700], v[perm]) and np.array_equal(n2[:700], n[perm])
    for i in range(0, 700, 97):  # alone
        a1, v1, n1 = _gpu(me[i:i + 1], opp[i:i + 1], depth[i:i + 1], keys[i:i + 1], 3, 8)
        assert (a1[0], v1[0], n1[0]) == (a[i], v[i], n[i])


def test_depth_zero_is_the_philox_rule():
    from oracle import minimax_ref as mr
    from oracle import pyoracle as po

    me, opp, _, keys = _set(8, 1000, 0, seed=5)
    depth = np.zeros(1000, np.uint8)
    a, v, nodes = _gpu(me, opp, depth, keys, 123456789, 8)
    masks = po.legal_mask(me, opp)
    for i in range(1000):
        m = int(masks[i])
        moves = [b for b in range(64) if (m >> b) & 1]
        ev = bin(int(me[i])).count("1") - bin(int(opp[i])).count("1")
        if moves:
            k = mr.random_move_index(123456789, int(keys[i]), bin(int(me[i]) | int(opp[i])).count("1"), len(moves))
            assert a[i] == moves[k], i
        assert v[i] == ev and nodes[i] == 1


def test_refusals():
    from betazero_b200 import _lib, minimax, players, tournament

    L, st = _lib.load(), _lib.stream_ptr()
    me, opp = _dev([0x0000000810000000]), _dev([0x0000001008000000])
    d, k = torch.zeros(1, dtype=torch.uint8, device="cuda"), torch.zeros(1, dtype=torch.int64, device="cuda")
    a, v, n = (torch.empty(1, dtype=t, device="cuda") for t in (torch.uint8, torch.int8, torch.int64))
    ws = minimax.workspace(1)
    args = [_lib.dptr(x) for x in (me, opp, d, k)]
    outs = [_lib.dptr(ws), _lib.dptr(a), _lib.dptr(v), _lib.dptr(n)]
    assert L.bz_minimax_moves(*args, 0, 1, 8, *outs, st) == 0
    for bad_size in (0, 5, 7, 10):
        assert L.bz_minimax_moves(*args, 0, 1, bad_size, *outs, st) == -1
    assert L.bz_minimax_moves(*args, 0, -1, 8, *outs, st) == -1
    assert L.bz_minimax_moves(*args, 0, 1 << 25, 8, *outs, st) == -1
    assert L.bz_minimax_moves(None, *args[1:], 0, 1, 8, *outs, st) == -1
    assert L.bz_minimax_moves(*args, 0, 1, 8, None, *outs[1:], st) == -1
    assert L.bz_minimax_moves(*args, 0, 1, 8, ctypes.c_void_p(ws.data_ptr() + 8), *outs[1:], st) == -2
    for bad_depth in (-1, 9, 100):
        with pytest.raises(ValueError):
            minimax.best_moves(me, opp, bad_depth)
        with pytest.raises(ValueError):
            players.OptimalPlayer(1, bad_depth)
        with pytest.raises(ValueError):
            tournament.Minimax(bad_depth)
    with pytest.raises(ValueError):
        minimax.best_moves(me, opp, torch.tensor([9]))
    with pytest.raises(ValueError):
        minimax.best_moves(me, opp, 2, size=5)
    # the tournament entries refuse a bad depth table
    t = tournament.Tournament([tournament.Minimax(1), tournament.Minimax(2)], 4)
    t.init()
    t.layout()
    for table in ((1, 9), (-2, 1)):
        dt = (ctypes.c_int32 * 2)(*table)
        assert L.bz_tournament_minimax(t._ref, dt, _lib.dptr(t._minimax_ws), _lib.dptr(t.minimax_action), None, st) == -1
        assert L.bz_tournament_advance(t._ref, None, dt, _lib.dptr(t.minimax_action), st) == -1
    net_and_mm = (ctypes.c_int32 * 2)(-1, 2)  # a net entrant needs pools
    assert L.bz_tournament_advance(t._ref, None, net_and_mm, _lib.dptr(t.minimax_action), st) == -1
    assert L.bz_tournament_minimax(t._ref, t._depths, None, _lib.dptr(t.minimax_action), None, st) == -1


def test_players_in_the_arena_equal_the_definition():
    """OptimalPlayer / RandomPlayer in arena.play_game on oracle boards, against the definition replayed move for move"""
    from betazero_b200 import arena, players
    from oracle import minimax_ref as mr
    from oracle import pyoracle as po

    for size, (dx, do) in [(8, (2, 0)), (6, (3, 1)), (4, (8, 0)), (8, (0, 3))]:
        seed, key = 40 + size, 1000 + dx
        mk = {0: lambda s: players.RandomPlayer(s, size=size, seed=seed, game_key=key)}
        px = mk[0](1) if dx == 0 else players.OptimalPlayer(1, dx, size=size, seed=seed, game_key=key)
        po_ = mk[0](-1) if do == 0 else players.OptimalPlayer(-1, do, size=size, seed=seed, game_key=key)
        seen = []

        class Rec:
            def __init__(self, p):
                self.p = p

            def get_move(self, board):
                mv = self.p.get_move(board)
                seen.append((board.board.copy(), self.p.symbol, mv))
                return mv

        winner, counts, plies = arena.play_game(po.OracleReversiBoard, Rec(px), Rec(po_), size=size)
        assert len(seen) > 3
        for grid, sym, mv in seen:
            b = po.OracleReversiBoard(size=size)
            b.board = grid
            ref = mr.Minimax(sym, dx if sym == 1 else do, seed=seed, game_key=key)
            assert ref.get_move(b) == mv
        refx, refo = mr.Minimax(1, dx, seed=seed, game_key=key), mr.Minimax(-1, do, seed=seed, game_key=key)
        assert arena.play_game(po.OracleReversiBoard, refx, refo, size=size) == (winner, counts, plies)


def _replay(moves, opening, sides, K, size, seed, key):
    """one game on boards.ReversiBoard: the recorded opening, then alternating moves of each side's sequential player:
    sides = {1: entrant, -1: entrant}, an entrant (net, n_sims) or tournament.Minimax"""
    from betazero_b200 import boards, players, tournament

    def make(s, e):
        if isinstance(e, tournament.Minimax):
            return players.OptimalPlayer(s, e.depth, size=size, seed=seed, game_key=key)
        return players.MCTSPlayer(s, net=e[0], n_sims=e[1], size=size, n_leaves=K)

    board = boards.ReversiBoard(size=size)
    ps = {s: make(s, sides[s]) for s in (1, -1)}
    cur, seq = 1, []
    while not board.is_game_over():
        if len(seq) < opening:
            a = int(moves[len(seq)])
        elif board.generate_possible_moves(cur):
            r, c = ps[cur].get_move(board)
            a = r * 8 + c
        else:
            a = 64
        if a != 64:
            board = board.make_move(a >> 3, a & 7, cur)
        seq.append(a)
        cur = -cur
    winner, counts = board.get_score()
    return seq, winner, counts


def _check_replays(t, r, entrants, K, size, seed):
    for g in range(t.n_games):
        i, j = t.pairings[int(r["pairing"][g])]
        sides = {1: entrants[i], -1: entrants[j]} if g % 2 == 0 else {1: entrants[j], -1: entrants[i]}
        seq, winner, counts = _replay(r["moves"][g], t.opening_plies, sides, K, size, seed, g)
        n = len(seq)
        assert list(r["moves"][g][:n]) == seq and (r["moves"][g][n:] == 255).all(), g
        assert int(r["result"][g]) == winner and (int(r["count_x"][g]), int(r["count_o"][g])) == counts, g


@pytest.mark.parametrize("size,K", [(8, 1), (8, 4), (6, 1), (6, 4)])
def test_tournament_with_minimax_entrants_equals_sequential_players(size, K):
    from betazero_b200 import net, tournament

    a = net.make_net("mlp", seed=90 + size)
    entrants = [(a, 32), tournament.Minimax(2), tournament.Minimax(0)]
    seed = size * 10 + K
    t = tournament.Tournament(entrants, 4, n_leaves=K, board_size=size, seed=seed)
    r = t.play()
    assert r["finished"] == 12 and r["kinds"] == ["net", "minimax", "minimax"] and r["depths"] == [None, 2, 0]
    assert r["minimax_nodes"] > 0
    sims = sum(32 for g in range(12) for p in range(t.opening_plies, 128)
               if r["moves"][g][p] != 255 and (entrants[t.pairings[int(r["pairing"][g])][(g + p) % 2]] is entrants[0]))
    assert r["simulations"] == sims  # only net searches count
    _check_replays(t, r, entrants, K, size, seed)


def test_minimax_only_tournament_equals_its_replays_and_allocates_no_trees():
    from betazero_b200 import tournament

    entrants = [tournament.Minimax(3), tournament.Minimax(1), tournament.Minimax(0)]
    t = tournament.Tournament(entrants, 6, board_size=6, seed=7, first_pair_id=5)
    assert t.pools is None
    r = t.play()
    assert r["finished"] == 18 and r["simulations"] == 0 and r["minimax_nodes"] > 0
    # game keys count from 2 first_pair_id: replay with that offset
    for g in range(t.n_games):
        i, j = t.pairings[int(r["pairing"][g])]
        sides = {1: entrants[i], -1: entrants[j]} if g % 2 == 0 else {1: entrants[j], -1: entrants[i]}
        seq, winner, counts = _replay(r["moves"][g], t.opening_plies, sides, 4, 6, 7, 10 + g)
        assert list(r["moves"][g][:len(seq)]) == seq and int(r["result"][g]) == winner, g
    # a stronger search scores against depth 0
    assert r["ratings"][0] > r["ratings"][2]


def test_batched_match_against_minimax_and_layout_invariants():
    from betazero_b200 import match, net, tournament

    a, b = net.make_net("mlp", seed=31), net.make_net("mlp", seed=32)
    m = match.BatchedMatch(a, match.Minimax(1), 8, 16, board_size=6, seed=3)
    r = m.play()
    assert r["finished"] == 8 and r["wins"] + r["draws"] + r["losses"] == 8 and r["minimax_nodes"] > 0
    entrants = [(a, 16), tournament.Minimax(2), (b, 8), tournament.Minimax(0)]
    t = tournament.Tournament(entrants, 40, n_leaves=4, board_size=6, opening_plies=3, seed=4)
    for n in (a, b):
        n.prepare_inference()
    t.init()
    G = t.n_games
    g_idx = torch.arange(G)
    first, second = t.first.cpu().long()[g_idx // 2], t.second.cpu().long()[g_idx // 2]
    x_ent = torch.where(g_idx % 2 == 0, first, second)
    o_ent = torch.where(g_idx % 2 == 0, second, first)
    depths = torch.tensor([-1, 2, -1, 0])
    for _ in range(200):
        n_search, pad = t.layout()
        if n_search == 0:
            break
        res, player = t.result.cpu(), t.player.cpu()
        tog, got = t.tree_of_game.cpu(), t.game_of_tree.cpu()
        live = res == match.RUNNING
        assert len(set(tog[live].tolist())) == int(live.sum()) and torch.equal(got[tog[live].long()], g_idx[live].int())
        mover = torch.where(player > 0, x_ent, o_ent)
        tree_ent = t.pair_net.cpu().long().repeat_interleave(56)[:n_search]
        assert torch.equal(tree_ent[tog[live].long()], mover[live])
        assert t._net_moves == bool((depths[mover[live]] < 0).any()) and t._minimax_moves == bool((depths[mover[live]] >= 0).any())
        t.pools.arena_used.fill_(-7)  # marks what the reset does not rewrite
        t.search(n_search)
        t.minimax_search()
        torch.cuda.synchronize()
        is_mm = depths[tree_ent] >= 0
        used, sims = t.pools.arena_used.cpu()[:n_search], t.pools.sim_count.cpu()[:n_search]
        if t._net_moves:  # minimax trees: reset, then left alone (no simulations)
            assert (sims[is_mm] == 0).all() and (used[is_mm] != -7).all()
        if t._minimax_moves:
            act = t.minimax_action.cpu()[:n_search]
            assert (act[is_mm & (got[:n_search] >= 0)] <= 64).all() and (act[~is_mm | (got[:n_search] < 0)] == 255).all()
        t.advance()
    assert n_search == 0
    torch.cuda.synchronize()
    assert int(t._errors.item()) == 0


def test_loop_reports_eval_minimax():
    from betazero_b200 import loop

    args = loop.default_args(games=48, sims=16, leaves=4, plies=6, size=6, train_steps=2, batch=128, lr=1e-2,
                             iterations=1, eval_games=8, eval_minimax=1)
    lines = loop.run(args)
    e = lines[0]["eval_minimax"]
    assert e["depth"] == 1 and e["wins"] + e["draws"] + e["losses"] == 8 and e["minimax_nodes"] > 0
    with pytest.raises(ValueError):
        loop.LoopState(loop.default_args(games=48, sims=16, size=6, eval_minimax=2), 0, 1)
