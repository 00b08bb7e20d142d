"""Batched net-versus-net matches: bz_mcts_search_fused_entrants with two nets of equal budgets builds, for every CTA
pair, exactly the trees the single-net one-launch search builds with that pair's net; BatchedMatch plays the games
MCTSPlayer plays one at a time, independently of the batch around them, with a consistent per-ply tree layout."""
import ctypes

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _roots(B, seed, size=8):
    from betazero_b200 import env
    from oracle import pyoracle as po

    if size != 8:
        me, opp, _ = env.reversi_init(B, size)
        return me, opp
    me_h, opp_h = po.playout_boards(B, seed=seed)  # midgame positions, including forced passes and finished games
    return env.to_device_u64(me_h), env.to_device_u64(opp_h)


def _search(model, me, opp, n_sims, K, size=8, two=None):
    """one-launch search of the roots with `model`; two = (model_b, pair_net): bz_mcts_search_fused_entrants with the
    entrants (model, n_sims) and (model_b, n_sims)"""
    from betazero_b200 import _lib, mcts

    B = me.numel()
    s = mcts.BatchedMCTS(mcts.TreePools(B, n_sims, board_size=size, n_leaves=K), mcts.FusedNetEvaluator(model),
                         use_graph=False, one_launch=True)
    s.pools.arena.zero_()  # the padding words at the end of a node block are never written: make them comparable
    s.reset(me, opp)
    if two is None:
        s.run(n_sims)
    else:
        model_b, pair_net = two
        model_b.prepare_inference()
        images = (ctypes.c_void_p * 2)(model._image_pair.data_ptr(), model_b._image_pair.data_ptr())
        iters = (ctypes.c_int32 * 2)(n_sims // K, n_sims // K)
        _lib.check(_lib.load().bz_mcts_search_fused_entrants(s.pools._ref, images, iters, 2, _lib.dptr(pair_net),
                                                             _lib.stream_ptr()), "entrants")
    torch.cuda.synchronize()
    s.check_errors()
    return s


def _tree_state(s):
    """per-tree tensors [B, ...]: root edges, allocator state, the arena's live words (dead words zeroed)"""
    p = s.pools
    used = p.arena_used.long() * 8
    arena = p.arena.view(p.n_trees, -1)
    col = torch.arange(arena.shape[1], device=arena.device)[None, :]
    out = [x.clone() for x in s.root_edges()]
    out += [getattr(p, n)[: p.n_trees].clone() for n in ("arena_used", "edge_count", "sim_count", "depth_sum", "root_meta")]
    out.append(torch.where(col < used[:, None], arena, torch.zeros_like(arena)))
    return out


@pytest.mark.parametrize("K", [1, 2, 4])
@pytest.mark.parametrize("B", [56, 57, 300, 4144, 4145, 9000])  # above 4144 trees: chunks, one launch each
def test_two_entrant_search_equals_the_single_net_searches(B, K):
    from betazero_b200 import net

    a, b = net.make_net("mlp", seed=10 + B + K), net.make_net("mlp", seed=20 + B + K)
    me, opp = _roots(B, seed=B + K)
    n_sims = (64 if B <= 300 else 16) // K * K
    g = torch.Generator().manual_seed(B * 10 + K)
    n_pairs = -(-B // 56)
    pair_net = torch.randint(0, 2, (n_pairs,), generator=g, dtype=torch.uint8)
    pair_net[0] = 1
    if n_pairs > 1:
        pair_net[-1] = 0  # both nets present whenever there are two pairs
    sel_b = pair_net.repeat_interleave(56)[:B].bool().cuda()
    ref_a, ref_b = _tree_state(_search(a, me, opp, n_sims, K)), _tree_state(_search(b, me, opp, n_sims, K))
    got = _tree_state(_search(a, me, opp, n_sims, K, two=(b, pair_net.cuda())))
    for x, ya, yb in zip(got, ref_a, ref_b):
        sel = sel_b.view(-1, *([1] * (x.dim() - 1)))
        assert torch.equal(x, torch.where(sel, yb, ya))
    assert not torch.equal(ref_a[0], ref_b[0])  # the two nets search differently: the comparison can tell them apart


@pytest.mark.parametrize("size", [6, 4])
def test_two_entrant_search_small_boards(size):
    from betazero_b200 import net

    a, b = net.make_net("mlp", seed=31), net.make_net("mlp", seed=32)
    me, opp = _roots(300, 0, size=size)
    pair_net = torch.tensor([0, 1, 1, 0, 1, 0], dtype=torch.uint8)
    sel_b = pair_net.repeat_interleave(56)[:300].bool().cuda()
    ref_a, ref_b = _tree_state(_search(a, me, opp, 32, 4, size)), _tree_state(_search(b, me, opp, 32, 4, size))
    got = _tree_state(_search(a, me, opp, 32, 4, size, two=(b, pair_net.cuda())))
    for x, ya, yb in zip(got, ref_a, ref_b):
        assert torch.equal(x, torch.where(sel_b.view(-1, *([1] * (x.dim() - 1))), yb, ya))


def _match(a, b, n_games, n_sims, K=4, size=8, opening=4, seed=0):
    from betazero_b200 import match

    return match.BatchedMatch(a, b, n_games, n_sims, n_leaves=K, board_size=size, opening_plies=opening, seed=seed).play()


def test_a_net_against_itself_scores_exactly_one_half():
    from betazero_b200 import net

    a, b = net.make_net("mlp", seed=3), net.make_net("mlp", seed=3)  # two separately built copies of one net
    r = _match(a, b, 512, 32, K=4, seed=5)
    mv, res = r["moves"], r["result"]
    assert np.array_equal(mv[0::2], mv[1::2])  # a pair's two games: the same moves ...
    assert np.array_equal(res[0::2], res[1::2])  # ... the same winner colour, i.e. opposite results for net A
    assert r["score"] == 0.5 and r["wins"] == r["losses"] and r["wins"] + r["draws"] + r["losses"] == 512
    assert r["disc_diff"] == 0 and r["elo"] == 0.0
    assert r["finished"] == 512 and (res != 2).all()
    assert r["plies"] > 20 and r["simulations"] > 0


def _replay(moves, opening, nets, n_sims, K, size):
    """one game on boards.ReversiBoard: the recorded opening, then alternating MCTSPlayer moves (arena.play_game's order)"""
    from betazero_b200 import boards, players

    board = boards.ReversiBoard(size=size)
    ps = {s: players.MCTSPlayer(s, net=nets[s], n_sims=n_sims, size=size, n_leaves=K) for s in (1, -1)}
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


@pytest.mark.parametrize("size,K", [(8, 1), (8, 4), (6, 1), (6, 4), (4, 4)])
def test_match_games_equal_sequential_mcts_player_games(size, K):
    from betazero_b200 import net

    a, b = net.make_net("mlp", seed=40 + size), net.make_net("mlp", seed=50 + size)
    r = _match(a, b, 16, 32, K=K, size=size, opening=4, seed=size * 10 + K)
    for g in range(16):
        nets = {1: a, -1: b} if g % 2 == 0 else {1: b, -1: a}
        seq, winner, counts = _replay(r["moves"][g], 4, nets, 32, K, size)
        n = len(seq)
        assert list(r["moves"][g][:n]) == seq and (r["moves"][g][n:] == 255).all(), g
        assert int(r["result"][g]) == winner and (int(r["count_x"][g]), int(r["count_o"][g])) == counts, g


def test_a_game_does_not_depend_on_the_batch_around_it():
    from betazero_b200 import net

    a, b = net.make_net("mlp", seed=61), net.make_net("mlp", seed=62)
    small = _match(a, b, 16, 8, K=4, seed=9)
    big = _match(a, b, 4200, 8, K=4, seed=9)  # 4255 trees: the early plies are searched in two chunks
    assert np.array_equal(small["moves"], big["moves"][:16]) and np.array_equal(small["result"], big["result"][:16])
    assert big["finished"] == 4200 and big["wins"] + big["draws"] + big["losses"] == 4200


def test_layout_invariants_every_ply():
    from betazero_b200 import match, net

    a, b = net.make_net("mlp", seed=71), net.make_net("mlp", seed=72)
    m = match.BatchedMatch(a, b, 600, 16, n_leaves=4, board_size=6, opening_plies=3, seed=4)
    a.prepare_inference()
    b.prepare_inference()
    m.init()
    g_idx = torch.arange(600)
    saw_padding = False
    for _ in range(200):
        n_search, pad = m.layout()
        c = m.counters.cpu()
        res, player = m.result.cpu(), m.player.cpu()
        tog, got = m.tree_of_game.cpu(), m.game_of_tree.cpu()
        live = res == match.RUNNING
        assert int(c[0]) == int(live.sum()) and int(c[1]) == n_search and int(c[2]) == pad
        assert int(c[3]) == int((~live).sum()) == int(c[4] + c[5] + c[6])
        assert (tog[~live] == -1).all() and (tog[live] >= 0).all() and (tog[live] < n_search).all()
        assert len(set(tog[live].tolist())) == int(live.sum())  # one tree per live game
        assert torch.equal(got[tog[live].long()], g_idx[live].int())
        net_to_move = (g_idx & 1) ^ (player < 0).long()
        pn = m.pair_net.cpu()[: -(-n_search // 56)].long()
        tree_net = pn.repeat_interleave(56)[:n_search]
        assert torch.equal(tree_net[tog[live].long()], net_to_move[live])  # each 56-tree group: one net's movers
        is_pad = got[:n_search] == -1
        assert int(is_pad.sum()) == pad
        if pad:
            saw_padding = True
            assert (m.root_me.cpu()[:n_search][is_pad] == 0).all() and (m.root_opp.cpu()[:n_search][is_pad] == 0).all()
            assert (tree_net[is_pad] == 0).all()  # padding closes net A's range
        for k in (0, 1):  # stable: game order within each net's range
            gs = got[:n_search][(tree_net == k) & ~is_pad]
            assert (gs[1:] > gs[:-1]).all()
        if n_search == 0:
            break
        m.search(n_search)
        m.advance()
    assert n_search == 0 and saw_padding
    torch.cuda.synchronize()
    assert int(m._errors.item()) == 0


def test_edge_cases_openings_passes_and_refusals():
    from betazero_b200 import match, net

    a, b = net.make_net("mlp", seed=81), net.make_net("mlp", seed=82)
    # 4x4: every game ends inside a 40-ply opening -- scored there, no search at all
    r = _match(a, b, 64, 8, K=4, size=4, opening=40, seed=1)
    assert r["plies"] == 0 and r["finished"] == 64 and r["simulations"] == 0
    cx, co = r["count_x"].astype(int), r["count_o"].astype(int)
    assert np.array_equal(r["result"], np.sign(cx - co))
    assert np.array_equal(r["moves"][0::2], r["moves"][1::2])  # a pair's games share the opening
    assert (r["moves"] == 64).any()  # 4x4 games are full of forced passes
    # opening_plies = 0: every pair plays the same two games
    r = _match(a, b, 32, 8, K=2, size=6, opening=0)
    assert (r["moves"][0::2] == r["moves"][0]).all() and (r["moves"][1::2] == r["moves"][1]).all()
    assert r["wins"] + r["draws"] + r["losses"] == 32
    # forced passes inside the nets' part of 4x4 games
    r = _match(a, b, 256, 8, K=1, size=4, opening=1, seed=2)
    assert any(64 in row[1:] for row in r["moves"]) and r["finished"] == 256
    with pytest.raises(ValueError):
        match.BatchedMatch(a, b, 15, 8)
    with pytest.raises(ValueError):
        match.BatchedMatch(a, net.make_net("resnet"), 16, 8)
    with pytest.raises(ValueError):
        match.BatchedMatch(net.make_net("mlp", game="ttt"), b, 16, 8)
    with pytest.raises(ValueError):
        match.BatchedMatch(a, net.make_net("mlp", hidden=128), 16, 8)
    with pytest.raises(ValueError):
        match.BatchedMatch(a, b, 16, 12, n_leaves=3)


@pytest.mark.parametrize("leaves", [1, 4])
def test_loop_iteration_reports_an_evaluation_match(leaves):
    from betazero_b200 import loop

    args = loop.default_args(games=48, sims=16, leaves=leaves, plies=8, size=6, train_steps=2, batch=128, lr=1e-2,
                             temp_plies=30, eval_games=40)
    st = loop.LoopState(args, rank=0, world=1)
    line = loop.run_iteration(st, 0)
    ev = line["eval"]
    assert ev["wins"] + ev["draws"] + ev["losses"] == 40
    assert 0.0 <= ev["score"] <= 1.0 and len(ev["elo_ci"]) == 2 and ev["ms"] > 0
    assert "eval" not in loop.run_iteration(loop.LoopState(loop.default_args(games=48, sims=16, leaves=leaves, plies=2,
                                                                               size=6, train_steps=1, batch=64), 0, 1), 0)
