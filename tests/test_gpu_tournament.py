"""Batched round-robin tournaments: bz_mcts_search_fused_entrants builds, for every CTA pair, exactly the trees the
single-net one-launch search builds with that pair's net and budget; bz_tournament_layout keeps each entrant's movers in
its own pair-aligned range; Tournament plays the games MCTSPlayer plays one at a time with each side's own budget, and
each pairing equals a standalone BatchedMatch."""
import ctypes

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _roots(B, seed):
    from betazero_b200 import env
    from oracle import pyoracle as po

    me_h, opp_h = po.playout_boards(B, seed=seed)  # midgame positions, including forced passes and finished games
    return env.to_device_u64(me_h), env.to_device_u64(opp_h)


def _pools_search(me, opp, cap, K):
    """a BatchedMCTS over the roots, its pools sized for `cap` simulations, reset and not yet searched"""
    from betazero_b200 import mcts, net

    B = me.numel()
    s = mcts.BatchedMCTS(mcts.TreePools(B, cap, n_leaves=K), mcts.FusedNetEvaluator(net.make_net("mlp", seed=0)),
                         use_graph=False, one_launch=True)
    s.pools.arena.zero_()  # the padding words at the end of a node block are never written: make them comparable
    s.reset(me, opp)
    return s


def _entrants_call(s, images, iters, pair_entrant):
    from betazero_b200 import _lib

    L = _lib.load()
    E = len(images)
    return L.bz_mcts_search_fused_entrants(s.pools._ref, (ctypes.c_void_p * E)(*images), (ctypes.c_int32 * E)(*iters), E,
                                           _lib.dptr(pair_entrant), _lib.stream_ptr())


def _single(model, me, opp, n_sims, cap, K):
    """bz_mcts_search_fused of the roots with one net, in pools sized for `cap` simulations"""
    from betazero_b200 import _lib

    s = _pools_search(me, opp, cap, K)
    model.prepare_inference()
    _lib.check(_lib.load().bz_mcts_search_fused(s.pools._ref, _lib.dptr(model._image_pair), None, n_sims // K,
                                                _lib.stream_ptr()), "search_fused")
    torch.cuda.synchronize()
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
@pytest.mark.parametrize("B", [56, 300, 4145, 9000])  # above 4144 trees: chunks, one launch each
def test_entrant_search_equals_the_single_net_searches(B, K):
    from betazero_b200 import _lib, net

    a, b, c = (net.make_net("mlp", seed=100 + 10 * i + B + K) for i in range(3))
    budgets = [16, 32, 64, 32, 48] if B <= 300 else [8, 16, 24, 8, 16]
    models = [a, b, a, c, b]  # a and b each under two budgets
    E = 3 + (B + K) % 3  # 3 .. 5 entrants
    models, budgets = models[:E], budgets[:E]
    for m in models:
        m.prepare_inference()
    cap = max(budgets)
    me, opp = _roots(B, seed=B + K)
    n_pairs = -(-B // 56)
    g = torch.Generator().manual_seed(B * 10 + K)
    pair_entrant = torch.randint(0, E, (n_pairs,), generator=g, dtype=torch.uint8)
    if n_pairs >= E:
        pair_entrant[:E] = torch.randperm(E, generator=g).to(torch.uint8)  # every entrant present
    s = _pools_search(me, opp, cap, K)
    _lib.check(_entrants_call(s, [m._image_pair.data_ptr() for m in models], [x // K for x in budgets],
                              pair_entrant.cuda()), "entrants")
    torch.cuda.synchronize()
    s.check_errors()
    got = _tree_state(s)
    refs = [_tree_state(_single(m, me, opp, n, cap, K)) for m, n in zip(models, budgets)]
    tree_ent = pair_entrant.repeat_interleave(56)[:B].long().cuda()
    for f, x in enumerate(got):
        want = torch.stack([r[f] for r in refs])[tree_ent, torch.arange(B, device="cuda")]
        assert torch.equal(x, want), f
    assert not torch.equal(refs[0][0], refs[1][0])  # the entrants search differently: the comparison can tell them apart


def test_a_one_entry_table_equals_the_single_net_search():
    from betazero_b200 import _lib, net

    a = net.make_net("mlp", seed=7)
    a.prepare_inference()
    me, opp = _roots(300, seed=3)
    s = _pools_search(me, opp, 32, 4)
    _lib.check(_entrants_call(s, [a._image_pair.data_ptr()], [8], torch.zeros(6, dtype=torch.uint8, device="cuda")), "one")
    torch.cuda.synchronize()
    for x, y in zip(_tree_state(s), _tree_state(_single(a, me, opp, 32, 32, 4))):
        assert torch.equal(x, y)


def test_an_entrant_without_iterations_leaves_its_trees_as_reset():
    from betazero_b200 import _lib, net

    a = net.make_net("mlp", seed=8)
    a.prepare_inference()
    me, opp = _roots(224, seed=4)
    fresh = _tree_state(_pools_search(me, opp, 32, 4))
    s = _pools_search(me, opp, 32, 4)
    pe = torch.tensor([1, 0, 1, 0], dtype=torch.uint8, device="cuda")
    _lib.check(_entrants_call(s, [a._image_pair.data_ptr()] * 2, [8, 0], pe), "zero")
    torch.cuda.synchronize()
    ref = _tree_state(_single(a, me, opp, 32, 32, 4))
    idle = pe.repeat_interleave(56).bool()
    for x, f, r in zip(_tree_state(s), fresh, ref):
        assert torch.equal(x, torch.where(idle.view(-1, *([1] * (x.dim() - 1))), f, r))


def _tournament(entrants, gpp, K=4, size=8, opening=4, seed=0, pairings=None):
    from betazero_b200 import tournament

    return tournament.Tournament(entrants, gpp, n_leaves=K, board_size=size, opening_plies=opening, seed=seed,
                                 pairings=pairings)


def _replay(moves, opening, sides, K, size):
    """one game on boards.ReversiBoard: the recorded opening, then alternating MCTSPlayer moves, each side with its own
    net and budget: sides = {1: (net, n_sims), -1: (net, n_sims)}"""
    from betazero_b200 import boards, players

    board = boards.ReversiBoard(size=size)
    ps = {s: players.MCTSPlayer(s, net=sides[s][0], n_sims=sides[s][1], size=size, n_leaves=K) for s in (1, -1)}
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


@pytest.mark.parametrize("size,K", [(8, 1), (8, 4), (6, 1), (6, 4)])
def test_tournament_games_equal_sequential_mcts_player_games(size, K):
    from betazero_b200 import net

    a, b = net.make_net("mlp", seed=40 + size), net.make_net("mlp", seed=50 + size)
    entrants = [(a, 32), (b, 16), (a, 8)]  # unequal budgets; net a under two of them
    t = _tournament(entrants, 4, K=K, size=size, seed=size * 10 + K)
    r = t.play()
    assert r["finished"] == 12
    for g in range(12):
        i, j = t.pairings[int(r["pairing"][g])]
        sides = {1: entrants[i], -1: entrants[j]} if g % 2 == 0 else {1: entrants[j], -1: entrants[i]}
        seq, winner, counts = _replay(r["moves"][g], 4, sides, K, size)
        n = len(seq)
        assert list(r["moves"][g][:n]) == seq and (r["moves"][g][n:] == 255).all(), g
        assert int(r["result"][g]) == winner and (int(r["count_x"][g]), int(r["count_o"][g])) == counts, g


def test_each_pairing_equals_a_standalone_batched_match():
    from betazero_b200 import match, net

    nets = [net.make_net("mlp", seed=60 + i) for i in range(3)]
    r = _tournament([(n, 16) for n in nets], 8, seed=11).play()
    for k, (i, j) in enumerate([(0, 1), (0, 2), (1, 2)]):
        m = match.BatchedMatch(nets[i], nets[j], 8, 16, seed=11, first_pair_id=4 * k).play()
        sl = slice(8 * k, 8 * k + 8)
        assert np.array_equal(r["moves"][sl], m["moves"]) and np.array_equal(r["result"][sl], m["result"]), k
        p = r["pairings"][k]
        assert (p["wins"], p["draws"], p["losses"]) == (m["wins"], m["draws"], m["losses"])
        assert p["score"] == m["score"] and r["crosstable"][i][j] == m["score"]


def test_a_net_against_its_own_copies_scores_one_half_and_rates_zero():
    from betazero_b200 import net

    copies = [net.make_net("mlp", seed=3) for _ in range(4)]  # separately built copies of one net
    r = _tournament([(n, 16) for n in copies], 32, seed=5).play()
    assert r["finished"] == 6 * 32
    for p in r["pairings"]:
        assert p["score"] == 0.5 and p["wins"] == p["losses"]
    assert r["ratings"] == [0.0] * 4
    mv = r["moves"]
    assert np.array_equal(mv[0::2], mv[1::2])  # a pair's two games: the same moves
    assert r["plies"] > 20 and r["simulations"] > 0 and r["chunks_per_ply"] == 1


def test_layout_invariants_every_ply():
    from betazero_b200 import match, net

    a, b = net.make_net("mlp", seed=71), net.make_net("mlp", seed=72)
    entrants = [(a, 16), (b, 8), (a, 4), (b, 16), (a, 8)]
    t = _tournament(entrants, 40, K=4, size=6, opening=3, seed=4, pairings=[(0, 1), (2, 0), (1, 3), (4, 3), (2, 4)])
    for n in (a, b):
        n.prepare_inference()
    G = t.n_games
    t.init()
    g_idx = torch.arange(G)
    first, second = t.first.cpu().long()[g_idx // 2], t.second.cpu().long()[g_idx // 2]
    x_ent = torch.where(g_idx % 2 == 0, first, second)
    o_ent = torch.where(g_idx % 2 == 0, second, first)
    saw_padding = False
    for _ in range(200):
        n_search, pad = t.layout()
        c = t.counters.cpu()
        res, player = t.result.cpu(), t.player.cpu()
        tog, got = t.tree_of_game.cpu(), t.game_of_tree.cpu()
        live = res == match.RUNNING
        assert int(c[0]) == int(live.sum()) and int(c[1]) == n_search and int(c[2]) == pad
        assert int(c[3]) == int((~live).sum()) == int(c[4] + c[5] + c[6])
        assert (tog[~live] == -1).all() and (tog[live] >= 0).all() and (tog[live] < n_search).all()
        assert len(set(tog[live].tolist())) == int(live.sum())  # one tree per live game ...
        assert torch.equal(got[tog[live].long()], g_idx[live].int())  # ... and game_of_tree is its inverse
        assert int((got[:n_search] >= 0).sum()) == int(live.sum())
        mover = torch.where(player > 0, x_ent, o_ent)
        pe = t.pair_net.cpu()[: -(-n_search // 56)].long()
        tree_ent = pe.repeat_interleave(56)[:n_search]
        assert torch.equal(tree_ent[tog[live].long()], mover[live])  # each 56-tree pair: one entrant's movers
        is_pad = got[:n_search] == -1
        assert int(is_pad.sum()) == pad
        assert (t.root_me.cpu()[:n_search][is_pad] == 0).all() and (t.root_opp.cpu()[:n_search][is_pad] == 0).all()
        assert (tree_ent[1:] >= tree_ent[:-1]).all()  # entrants in id order
        present = sorted(set(mover[live].tolist()))
        expect_pad = 0
        for e in present:
            rows = (tree_ent == e).nonzero().flatten()
            n_e = int((mover[live] == e).sum())
            assert int(rows[0]) % 56 == 0  # every range starts on a pair boundary
            gs = got[:n_search][rows]
            assert torch.equal(gs[:n_e], g_idx[live & (mover == e)].int())  # the movers first, in game order ...
            assert (gs[n_e:] == -1).all()  # ... then the range's padding
            if e != present[-1]:
                assert len(rows) == -(-n_e // 56) * 56
                expect_pad += len(rows) - n_e
            else:
                assert len(rows) == n_e  # the last range is not padded
        assert pad == expect_pad
        saw_padding |= pad > 0
        if n_search == 0:
            break
        t.search(n_search)
        t.advance()
    assert n_search == 0 and saw_padding
    torch.cuda.synchronize()
    assert int(t._errors.item()) == 0


def test_refusals():
    from betazero_b200 import _lib, mcts, net, tournament

    a = net.make_net("mlp", seed=81)
    with pytest.raises(ValueError):
        tournament.Tournament([], 2)
    with pytest.raises(ValueError):
        tournament.Tournament([(a, 8)] * 65, 2)
    with pytest.raises(ValueError):
        tournament.Tournament([(a, 8), (a, 6)], 2, n_leaves=4)
    with pytest.raises(ValueError):
        tournament.Tournament([(a, 8), (a, 8)], 3)
    with pytest.raises(ValueError):
        tournament.Tournament([(a, 8), (a, 8)], 65536)
    with pytest.raises(ValueError):
        tournament.Tournament([(a, 8), (a, 8), (a, 8)], 2, pairings=[(0, 1), (1, 2), (2, 1)])
    with pytest.raises(ValueError):
        tournament.Tournament([(a, 8), (a, 8)], 2, pairings=[(1, 1), (0, 1)])
    with pytest.raises(ValueError):
        tournament.Tournament([(a, 8), (net.make_net("resnet"), 8)], 2)
    with pytest.raises(ValueError):
        tournament.Tournament([(a, 8), (net.make_net("mlp", hidden=128), 8)], 2)

    a.prepare_inference()
    img = a._image_pair.data_ptr()
    p = mcts.TreePools(112, 8, n_leaves=4, prior_mode=mcts.PRIOR_LOGITS_BF16, eval_stride=72)
    L, st = _lib.load(), _lib.stream_ptr()
    pe = torch.zeros(2, dtype=torch.uint8, device="cuda")
    imgs, its = (ctypes.c_void_p * 2)(img, img), (ctypes.c_int32 * 2)(2, 2)
    assert L.bz_mcts_search_fused_entrants(p._ref, None, its, 2, _lib.dptr(pe), st) == -1  # no image table
    assert L.bz_mcts_search_fused_entrants(p._ref, imgs, None, 2, _lib.dptr(pe), st) == -1  # no count table
    assert L.bz_mcts_search_fused_entrants(p._ref, imgs, its, 2, None, st) == -1  # no pair_entrant
    assert L.bz_mcts_search_fused_entrants(p._ref, imgs, its, 0, _lib.dptr(pe), st) == -1
    big_i, big_n = (ctypes.c_void_p * 65)(*[img] * 65), (ctypes.c_int32 * 65)(*[2] * 65)
    assert L.bz_mcts_search_fused_entrants(p._ref, big_i, big_n, 65, _lib.dptr(pe), st) == -1
    assert L.bz_mcts_search_fused_entrants(p._ref, (ctypes.c_void_p * 2)(img, None), its, 2, _lib.dptr(pe), st) == -1
    assert L.bz_mcts_search_fused_entrants(p._ref, imgs, (ctypes.c_int32 * 2)(2, -1), 2, _lib.dptr(pe), st) == -1
    assert L.bz_mcts_search_fused_entrants(p._ref, (ctypes.c_void_p * 2)(img, img + 8), its, 2, _lib.dptr(pe), st) == -2

    t = tournament.Tournament([(a, 8), (a, 8), (a, 8)], 4)
    s = _lib.BzTournamentState.from_buffer_copy(t.c_struct)
    s.first = None
    assert L.bz_tournament_layout(ctypes.byref(s), st) == -1
    s = _lib.BzTournamentState.from_buffer_copy(t.c_struct)
    s.match.n_trees = t.n_games + 55  # room for two entrants' padding, not three
    assert L.bz_tournament_layout(ctypes.byref(s), st) == -1
    s = _lib.BzTournamentState.from_buffer_copy(t.c_struct)
    s.n_entrants = 65
    assert L.bz_tournament_layout(ctypes.byref(s), st) == -1


def test_loop_keeps_every_iterations_checkpoint_and_they_play_a_tournament(tmp_path):
    from betazero_b200 import loop, train, tournament

    pattern = str(tmp_path / "it{iteration}.pt")
    args = loop.default_args(games=48, sims=16, leaves=4, plies=6, size=6, train_steps=2, batch=128, lr=1e-2,
                             iterations=2, checkpoint=pattern)
    lines = loop.run(args)
    paths = [str(tmp_path / "it0.pt"), str(tmp_path / "it1.pt")]
    assert [ln["checkpoint"] for ln in lines] == paths
    nets = [train.load_net(p) for p in paths]
    r = tournament.Tournament([(nets[0], 16), (nets[1], 16)], 8, board_size=6).play()
    assert r["finished"] == 8 and len(r["ratings"]) == 2 and r["ratings"][0] == 0.0
