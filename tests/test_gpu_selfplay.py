"""GPU: the lockstep self-play driver (bz_selfplay_*) against the oracle's sequential self-play,
replay-record integrity, Philox move sampling, symmetry augmentation and a training step."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import mcts_ref as mr  # noqa: E402
from oracle import pyoracle as po  # noqa: E402

pytestmark = pytest.mark.gpu


def _philox_ref(seed, gid, ply):
    M = 0xFFFFFFFF
    c = [gid & M, (gid >> 32) & M, ply & M, 0]
    k = [seed & M, (seed >> 32) & M]
    for _ in range(10):
        p0, p1 = 0xD2511F53 * c[0], 0xCD9E8D57 * c[2]
        c = [((p1 >> 32) ^ c[1] ^ k[0]) & M, p1 & M, ((p0 >> 32) ^ c[3] ^ k[1]) & M, p0 & M]
        k = [(k[0] + 0x9E3779B9) & M, (k[1] + 0xBB67AE85) & M]
    return c[0]


def test_philox_matches_python_restatement():
    from betazero_b200 import _lib

    gid = torch.tensor([0, 1, 2, 12345678901234, 4095, 7], dtype=torch.int64, device="cuda")
    ply = torch.tensor([0, 0, 5, 59, 127, 3], dtype=torch.int32, device="cuda")
    out = torch.zeros(6, dtype=torch.int32, device="cuda")
    seed = 0x1234567887654321
    _lib.check(_lib.load().bz_philox_u32(seed, _lib.dptr(gid), _lib.dptr(ply), _lib.dptr(out), 6, _lib.stream_ptr()))
    got = out.cpu().numpy().view(np.uint32)
    exp = [_philox_ref(seed, int(g), int(p)) for g, p in zip(gid.tolist(), ply.tolist())]
    assert got.tolist() == exp
    assert len(set(exp)) == 6


@pytest.mark.parametrize("size,n_sims,leaves", [(4, 24, 1), (6, 16, 1), (4, 24, 4), (6, 16, 2),
                                                (8, 32, 1), (8, 32, 4), (8, 64, 4), (8, 48, 2)])
def test_deterministic_selfplay_equals_sequential_oracle(size, n_sims, leaves):
    """temp_plies = 0 (always the most visited move): every slot plays the same game as the oracle's
    sequential self_play_game in the order of the reference loop; check records, z and restart.
    leaves > 1: the searches use virtual loss (wave mode on the GPU, MCTS.run_vl in the oracle).
    The 8x8 cases are the bench workload's board (BASELINE configs[3]): full 60-ply games, passes included."""
    from betazero_b200 import mcts, selfplay

    salt = 3
    game = mr.ReversiGame(po.OracleReversiBoard, size)
    hist, winner = mr.self_play_game(game, n_sims, 1.25, lambda a, b: mr.hash_eval(a, b, salt, 65), leaves=leaves)
    B = 5
    sp = selfplay.BatchedSelfPlay(B, n_sims, mcts.HashEvaluator(salt), board_size=size, temp_plies=0, use_graph=False,
                                  rank=1, world=3, n_leaves=leaves)
    assert sp.game_id.tolist() == [5, 6, 7, 8, 9]  # rank 1 of 3 owns ids rank*B + s
    for ply in range(len(hist)):
        assert sp.ply.tolist() == [ply] * B
        sp.play_move()
        assert sp.last_action.tolist() == [hist[ply][4]] * B
    sp.mcts.check_errors()
    st = sp.stats()
    assert st["games"] == B and st["plies"] == B * len(hist) and st["replay_records"] == B * len(hist)
    assert st[{1: "x_wins", -1: "o_wins", 0: "draws"}[winner]] == B and st["dropped"] == 0
    assert sp.ply.tolist() == [0] * B and sp.player.tolist() == [1] * B
    assert sp.game_id.tolist() == [5 + 15, 6 + 15, 7 + 15, 8 + 15, 9 + 15]  # id_stride = world * B
    rp = sp.drain_replay()
    assert rp["me"].numel() == B * len(hist)
    order = torch.argsort(rp["game"] * 1024 + rp["ply"].to(torch.int64))
    me = rp["me"][order].cpu().numpy().view(np.uint64).reshape(B, -1)
    opp = rp["opp"][order].cpu().numpy().view(np.uint64).reshape(B, -1)
    pi = rp["pi"][order].cpu().numpy().reshape(B, len(hist), 65)
    z = rp["z"][order].cpu().numpy().reshape(B, -1)
    for k, (hme, hopp, hpl, hcnt, hact) in enumerate(hist):
        assert (me[:, k] == hme).all() and (opp[:, k] == hopp).all()
        assert (z[:, k] == winner * hpl).all()
        exp_pi = mr.policy_from_counts(hcnt)
        assert np.array_equal(pi[0, k], exp_pi) and (pi[:, k] == pi[0, k]).all()
    assert sp.stats()["replay_records"] == 0


def test_sampled_moves_follow_philox_and_visit_counts():
    """temp_plies > 0: the sampled action is the first edge whose cumulative visit count exceeds
    floor(u32 * total / 2^32), with u32 = Philox(seed, game id, ply): recompute on the host."""
    from betazero_b200 import mcts, selfplay

    B, n_sims, seed = 64, 40, 99
    sp = selfplay.BatchedSelfPlay(B, n_sims, mcts.HashEvaluator(1), temp_plies=100, seed=seed, use_graph=False)
    for ply in range(6):
        gids = sp.game_id.tolist()
        sp.search()
        cnt = sp.mcts.root_policy()[0].cpu().numpy()
        sp.advance()
        act = sp.last_action.cpu().numpy()
        for s in range(B):
            total = int(cnt[s].sum())
            target = (_philox_ref(seed, gids[s], ply) * total) >> 32
            cum = np.cumsum(cnt[s])
            assert act[s] == int(np.argmax(cum > target)), (ply, s)
    # different game ids diverge
    assert len({tuple(r) for r in sp.hist_action.view(B, -1)[:, :6].tolist()}) > 4


def test_full_games_recycle_slots_and_fill_replay():
    """8x8, small search: play until every slot has finished at least one game; check invariants
    of the replay buffer against the env oracle."""
    from betazero_b200 import mcts, net, selfplay

    B = 96
    sp = selfplay.BatchedSelfPlay(B, 12, mcts.FusedNetEvaluator(net.make_net("mlp", seed=2)), temp_plies=60, seed=5,
                                  graph_unroll=4)
    sp.prepare()
    for _ in range(75):
        sp.play_move()
    sp.mcts.check_errors()
    st = sp.stats()
    assert st["games"] >= B and st["dropped"] == 0
    assert st["x_wins"] + st["o_wins"] + st["draws"] == st["games"]
    rp = sp.drain_replay()
    n = rp["me"].numel()
    assert n == st["replay_records"] and n >= B * 50
    me, opp = rp["me"].cpu().numpy().view(np.uint64), rp["opp"].cpu().numpy().view(np.uint64)
    pi, z = rp["pi"].cpu().numpy(), rp["z"].cpu().numpy()
    assert not (me & opp).any()
    np.testing.assert_allclose(pi.sum(1), 1.0, atol=1e-5)
    mask = po.legal_mask(me, opp)
    legal = ((mask[:, None] >> np.arange(64, dtype=np.uint64)) & np.uint64(1)).astype(bool)
    assert (pi[:, :64][~legal] == 0).all()  # no probability on illegal cells
    assert ((pi[:, 64] > 0) == (mask == 0)).all()  # pass exactly when there is no move
    assert set(np.unique(z)) <= {-1, 0, 1}
    # per game: ply 0 is the start position, z flips sign with the mover along the game
    g0 = rp["game"].cpu().numpy()
    first = rp["ply"].cpu().numpy() == 0
    assert (me[first] == np.uint64((1 << 27) | (1 << 36))).all()
    assert len(np.unique(g0)) == st["games"]


def test_replay_overflow_drops_whole_games_and_never_returns_unwritten_rows():
    """replay_cap too small for the finished games: a game either gets all of its rows or none (counted as dropped);
    drain_replay() warns and returns only rows some game really wrote"""
    from betazero_b200 import mcts, selfplay

    B, cap = 48, 100
    sp = selfplay.BatchedSelfPlay(B, 8, mcts.HashEvaluator(2), board_size=4, temp_plies=30, seed=3, use_graph=False,
                                  replay_cap=cap)
    sp.rp_me.fill_(-1)  # poison: an unwritten row would show up as me == opp == all ones
    sp.rp_opp.fill_(-1)
    sp.rp_pi.fill_(float("nan"))
    for _ in range(14):  # 4x4 games last <= 12 plies + passes
        sp.play_move()
    st = sp.stats()
    assert st["games"] >= B and st["dropped"] > 0
    assert st["replay_records"] <= cap
    with pytest.warns(RuntimeWarning, match="replay buffer overflow"):
        rp = sp.drain_replay()
    n = rp["me"].numel()
    assert n == st["replay_records"] and 0 < n <= cap
    me, opp = rp["me"].cpu().numpy().view(np.uint64), rp["opp"].cpu().numpy().view(np.uint64)
    assert not (me & opp).any()
    np.testing.assert_allclose(rp["pi"].cpu().numpy().sum(1), 1.0, atol=1e-5)
    game, ply = rp["game"].cpu().numpy(), rp["ply"].cpu().numpy()
    for g in np.unique(game):  # whole games only: plies 0 .. k-1 of every game present
        p = np.sort(ply[game == g])
        assert np.array_equal(p, np.arange(len(p)))


def test_symmetry_kernel_matches_reference_transform_list():
    """the dihedral transforms of the reference's dataset expansion (SL/train.py:27-36)"""
    from betazero_b200 import env, train

    tf = [lambda x: x, lambda x: x.flip(dims=[0]), lambda x: x.flip(dims=[1]), lambda x: x.rot90(1, [0, 1]),
          lambda x: x.rot90(2, [0, 1]), lambda x: x.rot90(3, [0, 1]), lambda x: x.t(),
          lambda x: x.flip(dims=[0]).flip(dims=[1]).t()]  # 7: anti-transpose (see include/betazero_b200.h)
    rng = np.random.default_rng(0)
    for size in (8, 6, 4):
        n = 64
        grid = rng.integers(-1, 2, size=(n, size, size))
        pig = rng.random((n, size, size)).astype(np.float32)
        me = np.zeros(n, np.uint64)
        opp = np.zeros(n, np.uint64)
        pi = np.zeros((n, 65), np.float32)
        for i in range(n):
            m, o = po.grid_to_wire(grid[i], 1)
            me[i], opp[i] = m, o
            for r in range(size):
                for c in range(size):
                    pi[i, r * 8 + c] = pig[i, r, c]
            pi[i, 64] = 0.25
        sym = (np.arange(n) % 8).astype(np.uint8)
        mo, oo, po_ = train.augment(env.to_device_u64(me), env.to_device_u64(opp), torch.from_numpy(pi).cuda(),
                                    torch.from_numpy(sym).cuda(), size)
        mo, oo, po_ = env.to_host_u64(mo), env.to_host_u64(oo), po_.cpu().numpy()
        for i in range(n):
            eg = tf[sym[i]](torch.from_numpy(grid[i])).numpy()
            ep = tf[sym[i]](torch.from_numpy(pig[i])).numpy()
            assert np.array_equal(po.wire_to_grid(mo[i], oo[i], size), eg)
            for r in range(size):
                for c in range(size):
                    assert po_[i, r * 8 + c] == ep[r, c]
            assert po_[i, 64] == np.float32(0.25)


def test_training_step_reduces_loss_on_selfplay_records():
    from betazero_b200 import mcts, net, selfplay, train

    model = net.make_net("mlp", seed=0, dtype=torch.float32)
    sp = selfplay.BatchedSelfPlay(64, 8, mcts.NetEvaluator(model), temp_plies=60, seed=1, use_graph=False, board_size=6)
    for _ in range(40):
        sp.play_move()
    rp = sp.drain_replay()
    assert rp["me"].numel() > 500
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)  # the reference's optimiser family (SL/train.py:87)
    idx = torch.arange(min(1024, rp["me"].numel()), device="cuda")
    planes, pi, z = train.make_batch(rp, idx, size=6, augment_seed=0)
    first = train.train_step(model, opt, planes, pi, z)
    for _ in range(30):
        last = train.train_step(model, opt, planes, pi, z)
    assert last["loss"] < first["loss"]


def test_bench_dump_outputs_repeat_and_describe_the_last_timed_step(tmp_path):
    """bench.py --dump-outputs: two runs with the same arguments write identical arrays; pi is the root visit
    distribution, and past the sampled opening plies (temp_plies 8 < warm-up 2 + 8 timed steps) the move played is the
    most visited root action"""
    import json
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    runs = []
    for k in range(2):
        out = tmp_path / f"run{k}"
        p = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--games", "256", "--sims", "64", "--steps", "8",
                            "--warmup", "2", "--no-extra", "--no-iteration", "--no-cpu-baseline", "--scale-games", "0",
                            "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, p.stderr[-2000:]
        assert json.loads(p.stdout.strip().splitlines()[-1])["steps"] == 8
        runs.append({f[:-4]: np.load(out / f) for f in sorted(os.listdir(out))})
    a, b = runs
    assert sorted(a) == ["action", "board", "counters", "player", "ply", "root_pi", "root_q", "root_visits"]
    for k in a:
        assert a[k].dtype in (np.float32, np.float64) and np.array_equal(a[k], b[k], equal_nan=True), k
    n = a["root_visits"]
    assert n.shape == (256, 65) and a["board"].shape == (256, 64)
    np.testing.assert_allclose(a["root_pi"], n / n.sum(1, keepdims=True), rtol=1e-6)
    late = a["ply"] >= 9  # searched at ply 8 or later (a game that ended restarts at ply 0)
    assert late.sum() > 200 and np.array_equal(a["action"][late], n[late].argmax(1).astype(np.float32))
    assert (a["board"][:, [27, 28, 35, 36]] != 0).all() and a["counters"][1] == 10 * 256  # centre cells; plies played
