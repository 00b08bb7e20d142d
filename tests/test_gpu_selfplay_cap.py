"""GPU: self-play with randomized search budgets (BatchedSelfPlay(fast_sims=n, full_fraction=p); bz_selfplay_cap_layout,
bz_selfplay_advance_cap, bz_selfplay_endgame_play_cap, bz_mcts_root_noise_entrant) against the sequential restatement
(oracle/selfplay_cap_ref.py) with the exactly representable nets of test_net_exact, against single-budget searches of the
same roots, and against self-play without the option."""
import ctypes

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import endgame_wld_ref as ewr  # noqa: E402
from oracle import mcts_ref as mr  # noqa: E402
from oracle import pyoracle as po  # noqa: E402
from oracle import selfplay_cap_ref as scr  # noqa: E402
from oracle import selfplay_endgame_ref as ser  # noqa: E402
from oracle import selfplay_resign_ref as srr  # noqa: E402
from test_net_exact import exact_net, walk_trees  # noqa: E402

pytestmark = pytest.mark.gpu
META_N_SHIFT = 7  # BZ_META_N_SHIFT


@pytest.fixture(scope="module", autouse=True)
def _selfplay_bounds_checks():
    """a -DBZ_BOUNDS_CHECK library: the violation record of the self-play kernels must stay empty"""
    yield
    from betazero_b200 import _lib

    if _lib._lib is not None and hasattr(_lib._lib, "bz_debug_checks_selfplay"):
        torch.cuda.synchronize()
        rec = (ctypes.c_int * 4)()
        assert _lib._lib.bz_debug_checks_selfplay(rec) == 0
        assert rec[3] == 0, f"check {rec[0]} failed in block {rec[1]}, thread {rec[2]} ({rec[3]} violations)"


@pytest.fixture(scope="module")
def net():
    m = exact_net(21, device="cuda")
    m.prepare_inference()
    return m


def _ev(net):
    from betazero_b200 import mcts

    return mcts.FusedNetEvaluator(net, use_kernel=True)


def _games(rp):
    """game id -> (me, opp, pi, z, full, q or None) in ply order; every game's plies are 0 .. n-1"""
    game, ply = rp["game"].cpu().numpy(), rp["ply"].cpu().numpy()
    cols = [rp["me"].cpu().numpy().view(np.uint64), rp["opp"].cpu().numpy().view(np.uint64), rp["pi"].cpu().numpy(),
            rp["z"].cpu().numpy(), rp["full"].cpu().numpy() if "full" in rp else None,
            rp["q"].cpu().numpy() if "q" in rp else None]
    out = {}
    order = np.lexsort((ply, game))
    for idx in np.split(order, np.flatnonzero(np.diff(game[order])) + 1):
        if idx.size:
            assert np.array_equal(ply[idx], np.arange(idx.size))
            out[int(game[idx[0]])] = tuple(None if c is None else c[idx] for c in cols)
    return out


class _TreeSearch:
    """the search of one fresh tree: a single-tree bz_mcts_search_fused, which every tree of the batched search equals"""

    def __init__(self, net, game, n_max, K):
        from betazero_b200 import mcts

        self.game, self.K, self.cache = game, K, {}
        self.m = mcts.BatchedMCTS(mcts.TreePools(1, n_max, board_size=game.size, n_leaves=K), _ev(net), use_graph=False,
                                  one_launch=True)

    def __call__(self, board, player, n):
        me, opp = self.game.wire(board, player)
        key = (me, opp, n)
        if key not in self.cache:
            t = torch.from_numpy(np.array([me, opp], np.uint64).view(np.int64)).cuda()
            self.m.reset(t[:1], t[1:])
            self.m.search_one_launch(n // self.K)
            N, W, _ = self.m.root_edges()
            self.cache[key] = (N[0].cpu().numpy(), W[0].cpu().numpy())
        return self.cache[key]


CASES = [  # size, K, n_sims, fast_sims, endgame_empties, solve, resign threshold
    (4, 1, 32, 8, 0, "exact", None), (4, 4, 32, 8, 6, "wld", 0.0), (4, 2, 16, 4, 6, "exact", None),
    (6, 2, 32, 8, 10, "exact", None), (6, 4, 48, 16, 0, "exact", 0.0), (6, 1, 32, 8, 10, "wld", 0.0),
    (8, 1, 32, 8, 0, "exact", None), (8, 2, 32, 8, 10, "wld", None), (8, 4, 64, 16, 10, "exact", 0.0),
    (8, 4, 32, 8, 0, "exact", -0.5),
]


@pytest.mark.parametrize("size,K,n_sims,fast,empties,solve,thr", CASES)
def test_records_equal_the_sequential_restatement(net, size, K, n_sims, fast, empties, solve, thr):
    """boards, pi, actions, z, game ids, q and flags of every finished game, bit for bit"""
    from betazero_b200 import selfplay

    B, seed, p, temp, audit = 8, 17, 0.5, 6, 0.3
    plies = {4: 24, 6: 44, 8: 76}[size]
    sp = selfplay.BatchedSelfPlay(B, n_sims, _ev(net), board_size=size, temp_plies=temp, seed=seed, n_leaves=K,
                                  use_graph=False, rank=1, world=2, endgame_empties=empties, endgame_every=1,
                                  endgame_solve=solve, resign_threshold=thr, resign_audit=audit, fast_sims=fast,
                                  full_fraction=p)
    for _ in range(plies):
        sp.play_move()
    sp.mcts.check_errors()
    st = sp.stats()
    got = _games(sp.drain_replay())
    assert len(got) >= B // 2 and st["dropped"] == 0
    assert st["full_plies"] > 0 and st["fast_plies"] > 0 and st["full_plies"] + st["fast_plies"] == B * plies
    game = mr.ReversiGame(po.OracleReversiBoard, size)
    search = _TreeSearch(net, game, n_sims, K)
    solver = ser.c_solver(game) if solve == "exact" else ewr.wld_solver(ser.c_solver(game))
    below, abelow = scr.full_below(p), srr.audit_below(audit)
    fast_rows = 0
    for g, (me, opp, pi, z, full, q) in got.items():
        assert g % B in range(B) and (g // B) % 2 == 1  # rank 1 of 2: ids B + s + 2 B k
        hist, winner, _, _ = scr.self_play_game_cap(game, n_sims, fast, search, seed, g, below, temp_plies=temp,
                                                    threshold=thr, is_audited=srr.audited(seed, g, abelow),
                                                    endgame_empties=empties, solve=solver)
        assert len(me) == len(hist), g
        for k, (hme, hopp, hpl, hpi, _, hq, hfull) in enumerate(hist):
            assert me[k] == hme and opp[k] == hopp and z[k] == winner * hpl and full[k] == hfull, (g, k)
            assert np.array_equal(pi[k], hpi), (g, k)
            if thr is not None:
                assert np.array_equal(q[k], hq, equal_nan=True), (g, k)
        fast_rows += int((full == 0).sum())
    assert fast_rows > 0


def _slot_trees(sp, ref_pools, t_of_s, walks=None):
    """slot s's tree of the self-play pools against tree s of ref_pools, for the slots in t_of_s ([k, 2]: slot, tree;
    both columns ascending): the per-tree counters, and every node the trees hold (walk_trees: board, edges, statistics,
    priors; the words of a node block past its edges are never read and are not compared)"""
    P, R = sp.pools, ref_pools
    for name in ("root_meta", "arena_used", "sim_count", "edge_count", "depth_sum", "error"):
        assert torch.equal(getattr(P, name)[t_of_s[:, 1]], getattr(R, name)[t_of_s[:, 0]]), name
    a, b = walks if walks is not None else (walk_trees(P), walk_trees(R))
    slots, trees = t_of_s[:, 0].cpu().numpy(), t_of_s[:, 1].cpu().numpy()
    slot_of_tree = np.full(P.n_trees, -1)
    slot_of_tree[trees] = slots
    sa, sb = np.isin(a["tree"], trees), np.isin(b["tree"], slots)
    assert sa.sum() == sb.sum() > 0
    for k in a:
        x, y = a[k][sa], b[k][sb]
        if k == "tree":
            x = slot_of_tree[x]
        if x.dtype.kind == "f":
            x, y = x.view(np.uint32), y.view(np.uint32)
        assert np.array_equal(x, y), k


@pytest.mark.parametrize("B,K,n_sims,fast,size", [(300, 1, 32, 8, 8), (500, 2, 32, 16, 6), (9000, 4, 16, 8, 8)])
def test_every_tree_equals_a_single_budget_search_of_its_root(net, B, K, n_sims, fast, size):
    """several plies; 9000 games: 9055 trees in three launches of the one-launch search"""
    from betazero_b200 import mcts, selfplay

    sp = selfplay.BatchedSelfPlay(B, n_sims, _ev(net), board_size=size, temp_plies=30, seed=3, n_leaves=K,
                                  use_graph=False, fast_sims=fast, full_fraction=0.3)
    refs = {n: mcts.BatchedMCTS(mcts.TreePools(B, n_sims, board_size=size, n_leaves=K), _ev(net), use_graph=False,
                                one_launch=True) for n in (n_sims, fast)}
    for ply in range(7):
        full = selfplay.is_full(sp.game_id, sp.ply, 3, 0.3)
        sp.search()
        torch.cuda.synchronize()
        t = sp.tree_of_slot.long()
        walk = walk_trees(sp.pools)
        for n, m in refs.items():
            m.reset(sp.me, sp.opp)
            m.search_one_launch(n // K)
            sel = full if n == n_sims else ~full
            slots = torch.nonzero(sel).squeeze(1)
            assert slots.numel() > 0
            _slot_trees(sp, m.pools, torch.stack([slots, t[slots]], 1), (walk, walk_trees(m.pools)))
        sp.advance()
    sp.mcts.check_errors()


def _check_layout(sp, seed, p):
    from betazero_b200 import selfplay

    B, T = sp.n_games, sp.pools.n_trees
    full = selfplay.is_full(sp.game_id, sp.ply, seed, p).cpu().numpy()
    t = sp.tree_of_slot.cpu().numpy()
    n_full = int(full.sum())
    fast0 = -(-n_full // 56) * 56
    assert np.array_equal(t[full], np.arange(n_full))  # stable: slot order inside each range
    assert np.array_equal(t[~full], fast0 + np.arange(B - n_full))
    assert fast0 % 56 == 0 and len(set(t.tolist())) == B  # a bijection onto the used trees
    pe = sp.pair_entrant.cpu().numpy()
    assert np.array_equal(pe, (np.arange(pe.size) * 56 >= fast0).astype(np.uint8))
    rm, ro = sp.cap_root_me.cpu().numpy(), sp.cap_root_opp.cpu().numpy()
    assert np.array_equal(rm[t], sp.me.cpu().numpy()) and np.array_equal(ro[t], sp.opp.cpu().numpy())
    pad = np.setdiff1d(np.arange(T), t)
    assert (rm[pad] == 0).all() and (ro[pad] == 0).all()
    meta = sp.pools.root_meta.cpu().numpy().view(np.uint32)
    assert (((meta[pad] >> META_N_SHIFT) & 63) == 0).all()  # padding trees are never expanded
    return n_full, pad


@pytest.mark.parametrize("p", [0.0, 0.25, 1.0])
def test_layout_invariants(net, p):
    from betazero_b200 import selfplay

    B = 700
    sp = selfplay.BatchedSelfPlay(B, 16, _ev(net), board_size=6, temp_plies=20, seed=5, n_leaves=4, use_graph=False,
                                  fast_sims=8, full_fraction=p)
    for ply in range(5):
        sp.search()
        n_full, pad = _check_layout(sp, 5, p)
        if p in (0.0, 1.0):
            assert n_full == (B if p == 1.0 else 0) and (pad >= B).all()  # no padding between the ranges
        else:
            assert 0 < n_full < B
        sp.advance()


@pytest.mark.parametrize("K,fast,p", [(1, 32, 0.3), (4, 8, 1.0), (2, 32, 0.6)])
def test_identities_against_self_play_without_the_option(net, K, fast, p):
    """p = 1: the same games, every flag 1; fast_sims == n_sims: the same games, the flags of the draw"""
    from betazero_b200 import selfplay

    kw = dict(board_size=6, temp_plies=10, seed=8, n_leaves=K, use_graph=False)
    off = selfplay.BatchedSelfPlay(128, 32, _ev(net), one_launch=True, **kw)
    on = selfplay.BatchedSelfPlay(128, 32, _ev(net), fast_sims=fast, full_fraction=p, **kw)
    for _ in range(50):
        off.play_move()
        on.play_move()
    a, b = _games(off.drain_replay()), _games(on.drain_replay())
    assert sorted(a) == sorted(b) and len(a) >= 128
    ids, plies = [], []
    for g in a:
        assert all(np.array_equal(x, y) for x, y in zip(a[g][:4], b[g][:4])), g
        ids += [g] * len(b[g][0])
        plies += list(range(len(b[g][0])))
    flags = np.concatenate([b[g][4] for g in a])
    want = selfplay.is_full(torch.tensor(ids), torch.tensor(plies), 8, p).cpu().numpy()
    assert np.array_equal(flags, want.astype(np.uint8))
    assert (p < 1.0) or flags.all()


def test_flag_frequency_and_counters(net):
    from betazero_b200 import selfplay

    B, p, seed = 2048, 0.25, 13
    sp = selfplay.BatchedSelfPlay(B, 16, _ev(net), board_size=6, temp_plies=40, seed=seed, n_leaves=4, use_graph=False,
                                  fast_sims=8, full_fraction=p)
    expect = 0
    for _ in range(40):
        expect += int(selfplay.is_full(sp.game_id, sp.ply, seed, p).sum())
        sp.play_move()
    st = sp.stats()
    n = B * 40
    assert st["full_plies"] == expect and st["fast_plies"] == n - expect
    assert abs(expect / n - p) < 5 * (p * (1 - p) / n) ** 0.5
    rp = sp.drain_replay()
    flags = rp["full"]
    want = selfplay.is_full(rp["game"], rp["ply"].to(torch.int64), seed, p)
    assert torch.equal(flags.bool(), want) and 0 < int(flags.sum()) < flags.numel()
    # the draw of the library equals the restatement's Philox
    g, t = rp["game"][:500].cpu().tolist(), rp["ply"][:500].cpu().tolist()
    assert want[:500].cpu().tolist() == [scr.is_full(seed, a, b, scr.full_below(p)) for a, b in zip(g, t)]


def test_root_noise_perturbs_full_trees_only(net):
    from betazero_b200 import mcts, selfplay

    B, K = 400, 4
    sp = selfplay.BatchedSelfPlay(B, 32, _ev(net), board_size=8, temp_plies=30, seed=4, n_leaves=K, use_graph=False,
                                  fast_sims=16, full_fraction=0.5, dirichlet_alpha=0.3)
    for _ in range(4):
        sp.play_move()
    full = selfplay.is_full(sp.game_id, sp.ply, 4, 0.5)
    sp.search()
    torch.cuda.synchronize()
    t = sp.tree_of_slot.long()
    _, _, P = sp.mcts.root_edges()
    for n, sel in ((32, full), (16, ~full)):
        m = mcts.BatchedMCTS(mcts.TreePools(B, 32, board_size=8, n_leaves=K), _ev(net), use_graph=False, one_launch=True)
        m.reset(sp.me, sp.opp)
        m.search_one_launch(n // K)
        _, _, Pr = m.root_edges()
        slots = torch.nonzero(sel).squeeze(1)
        differs = (P[t[slots]] != Pr[slots]).any(1)
        if n == 16:
            assert not differs.any()  # fast trees: no noise, the single-budget search exactly
            _slot_trees(sp, m.pools, torch.stack([slots, t[slots]], 1))
        else:
            assert differs.float().mean() > 0.9


def test_refusals(net):
    from betazero_b200 import _lib, mcts, selfplay

    L = _lib.load()
    with pytest.raises(ValueError, match="one-launch"):
        selfplay.BatchedSelfPlay(8, 16, mcts.HashEvaluator(1), fast_sims=8)
    with pytest.raises(ValueError, match="tree reuse"):
        selfplay.BatchedSelfPlay(8, 16, _ev(net), fast_sims=8, reuse=True)
    for empties in (0, 10):
        sp = selfplay.BatchedSelfPlay(8, 16, _ev(net), board_size=6, use_graph=False, endgame_empties=empties,
                                      resign_threshold=-1.0, fast_sims=8)
        sp.search()
        cs, eg = sp.cs, (sp._eg_ref if sp.eg is not None else None)

        def calls():
            st = _lib.stream_ptr()
            out = [L.bz_selfplay_cap_layout(sp._ref, sp._cs_ref, st),
                   L.bz_selfplay_advance_cap(sp._ref, eg, sp._rs_ref, sp._cs_ref, sp.pools._ref, None, st)]
            if empties:
                out.append(L.bz_selfplay_endgame_play_cap(sp._ref, eg, sp._rs_ref, sp._cs_ref,
                                                          _lib.dptr(sp.eg_workspace), 1, st))
            return out

        bad = [("full_below", (1 << 32) + 1), ("n_trees", 8 + 54), ("tree_of_slot", None), ("root_me", None),
               ("root_opp", None), ("pair_entrant", None), ("hist_full", None), ("rp_full", None), ("counters", None)]
        for field, value in bad:
            old = getattr(cs, field)
            setattr(cs, field, value)
            assert calls() == [-1] * len(calls()), field
            setattr(cs, field, old)
        if empties:
            old, cs.eg_hist_full = cs.eg_hist_full, None
            assert L.bz_selfplay_cap_layout(sp._ref, sp._cs_ref, _lib.stream_ptr()) == 0  # the layout has no queue
            assert calls()[1:] == [-1, -1]
            cs.eg_hist_full = old
            assert L.bz_selfplay_endgame_play_cap(sp._ref, eg, None, None, _lib.dptr(sp.eg_workspace), 0,
                                                  _lib.stream_ptr()) == -1
        assert L.bz_selfplay_cap_layout(sp._ref, None, _lib.stream_ptr()) == -1
        assert L.bz_selfplay_advance_cap(sp._ref, eg, None, None, sp.pools._ref, None, _lib.stream_ptr()) == -1
        # the pools must be the layout's: n_games + 55 trees
        small = mcts.TreePools(8, 16, board_size=6, n_leaves=1)
        assert L.bz_selfplay_advance_cap(sp._ref, eg, None, sp._cs_ref, small._ref, None, _lib.stream_ptr()) == -1
        cs.full_below = 1 << 32  # every ply full: accepted
        sp.search()
        assert calls()[1:] == [0] * (len(calls()) - 1)
        torch.cuda.synchronize()
    noise = torch.ones((sp.pools.n_trees, 65), device="cuda")
    assert L.bz_mcts_root_noise_entrant(sp.pools._ref, _lib.dptr(noise), 0.25, None, 0, _lib.stream_ptr()) == -1
    assert L.bz_mcts_root_noise_entrant(sp.pools._ref, None, 0.25, _lib.dptr(sp.pair_entrant), 0, _lib.stream_ptr()) == -1
    assert L.bz_mcts_root_noise_entrant(sp.pools._ref, _lib.dptr(noise), 1.5, _lib.dptr(sp.pair_entrant), 0,
                                        _lib.stream_ptr()) == -1


def test_loop_trains_on_full_records_only(tmp_path):
    from betazero_b200 import loop

    ck = str(tmp_path / "ck.pt")
    args = loop.default_args(games=256, sims=16, leaves=4, plies=70, train_steps=2, batch=256, lr=1e-3, size=6,
                             fast_sims=8, full_fraction=0.25, resign=-1.0, checkpoint=ck)
    (line,) = loop.run(args)
    cap = line["cap"]
    assert cap["full_fraction"] == 0.25 and cap["fast_sims"] == 8 and cap["games_finished_local"] > 0
    assert cap["full_plies_local"] + cap["fast_plies_local"] == 256 * 70 and cap["full_plies_local"] > 0
    n = line["replay_records_gathered"]
    assert 0 < cap["records_trained_on"] < n and line["train_batch"] == min(256, cap["records_trained_on"])
    assert "resign" in line and line["loss_first_last"] is not None
    extra = torch.load(ck, map_location="cpu", weights_only=True)["extra"]
    assert extra["fast_sims"] == 8 and extra["full_fraction"] == 0.25
    plain = loop.default_args(games=48, sims=16, plies=2, size=6, train_steps=1, batch=64)
    assert "cap" not in loop.run_iteration(loop.LoopState(plain, 0, 1), 0)
