"""The throughput path's priors and values, in every tree-kernel instantiation, against float64.

Every production search runs in BZ_PRIOR_LOGITS_BF16 mode: the tree kernel reads the net's bf16 row and computes the
legal-move softmax itself (exp_nonpos = ex2.approx.ftz, a group sum, __fdividef) and the value's tanhf.  That code is
written out four times in mcts.cu (the group kernels, the wave kernels and the one-launch search's two post-backup
routines) and instantiated per game, lane-group width, virtual-loss flag and kernel (step / expand_backup).

1. A board-keyed row evaluator: the bf16 row of a leaf is a pure function of its board, drawn from a palette of
   ordinary and edge-of-range rows (spreads past the flush, the maximum on an illegal column, ties, +-bf16 max,
   +-0 and subnormals; values that saturate tanh, +-0, subnormals).  The checker recomputes the row of every
   expanded node from the node's board, so colliding descents (K > 1) and every node of every tree are checked.
2. The instantiation matrix: Reversi 8x8 / 6x6 / 4x4 and tic-tac-toe, 8 / 16 / 32 lanes, wave mode and slots one after
   the other, the fused step and the unfused expand_backup kernels, and the dispatch's own choice at 8192 trees.
3. Tic-tac-toe with an exactly representable net (test_net_exact.py's construction on 9 signed inputs) through the
   library GEMMs: batched searches and TicTacToeMCTSPlayer in the reference's game loop.
4. The one-launch search with exact nets whose head is scaled by 2^40 (priors flushed, tanh saturated) and 2^-60
   (tiny logits and values), against float64 and against the per-iteration kernels.

NaN and +-inf logits are not in the palette: only a net whose fp32 accumulators overflowed produces them."""
import functools
import math

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from test_gpu_one_launch import _same_trees  # noqa: E402
from test_gpu_puct_edges import _fused_search  # noqa: E402
from test_net_exact import _roots as _net_roots  # noqa: E402
from test_net_exact import check_exact, check_search, exact_net, reference_forward, walk_trees  # noqa: E402

BF16_MAX = float(torch.finfo(torch.bfloat16).max)  # 3.3895e38
BF16_SUB = 2.0 ** -133  # the smallest bf16 subnormal
LOG2E = 1.4426950408889634
DC = abs(float(np.float32(LOG2E)) - LOG2E) / LOG2E + 2.0 ** -52  # relative error of fl(log2 e) (exp_nonpos)
PRIOR_KINDS = ("ordinary", "spread", "illegal-max", "all-equal", "bf16-max", "zero-subnormal")
VALUE_KINDS = ("ordinary", "zero", "subnormal", "saturated", "bf16-max")


# ---------------------------------------------------------------------------------------------------------------------
# the board-keyed rows
# ---------------------------------------------------------------------------------------------------------------------
def _i64(c):
    return c - (1 << 64) if c >= 1 << 63 else c


def _srl(x, s):
    """logical right shift of an int64 tensor"""
    return (x >> s) & ((1 << (64 - s)) - 1)


def _mix(x):
    """splitmix64's finaliser on int64 tensors (wrapping arithmetic)"""
    x = (x ^ _srl(x, 30)) * _i64(0xBF58476D1CE4E5B9)
    x = (x ^ _srl(x, 27)) * _i64(0x94D049BB133111EB)
    return x ^ _srl(x, 31)


def _uniform(h):
    """float64 in (0, 1) from the top 53 bits"""
    return (_srl(h, 11).double() + 0.5) * 2.0 ** -53


@torch.no_grad()
def board_rows(me, opp, A, stride):
    """(bf16 [n, stride] rows, prior kind [n], value kind [n]) of mover-relative boards (int64 tensors of uint64 bits):
    logits in columns 0..A-1, the pre-tanh value in column A, bf16 max in the padding columns (a kernel that read them
    as logits would take them for the maximum).  A 64-bit mix of the board picks the row's prior kind (PRIOR_KINDS),
    its value kind (VALUE_KINDS) and the per-cell values:
      ordinary        3 z (z standard normal)
      spread          -S u, S in [100, 300], u uniform: legal spreads past 87.3, where exp_nonpos flushes to 0
      illegal-max     3 z, and 30 + 3 |z| on every occupied cell and the pass column: the row's maximum is illegal
      all-equal       one value in every column: 3 z, 0, +bf16 max or -bf16 max
      bf16-max        3 z with 40 % of the cells +-bf16 max (w - m overflows to -inf where the maximum is +bf16 max)
      zero-subnormal  +-0 and +-k 2^-133 (bf16 subnormals)
    values: 2 z; +-0; +-k 2^-133; +-[10, 1000) (tanhf is exactly +-1); +-bf16 max."""
    n, dev = me.shape[0], me.device
    h = _mix(me ^ _mix(opp + 0x5DEECE66D))
    col = torch.arange(stride, device=dev, dtype=torch.int64)
    c1 = _mix(h[:, None] + col * _i64(0x9E3779B97F4A7C15))
    c2 = _mix(c1 ^ 0x2545F4914F6CDD1D)
    u1, u2 = _uniform(c1), _uniform(c2)
    z = torch.sqrt(-2.0 * torch.log(u1)) * torch.cos(2.0 * math.pi * u2)
    sign = torch.where((c2 & 1) == 1, -1.0, 1.0).double()
    sub = sign * (1 + _srl(c1, 40) % 127).double() * BF16_SUB
    hr = _uniform(_mix(h ^ 0x3C6EF372FE94F82B))[:, None]  # one uniform per row
    kind, vkind, pick = _srl(h, 8) % 6, _srl(h, 16) % 5, _srl(h, 24) % 4

    cells = min(A, 64)
    bits = torch.arange(cells, device=dev, dtype=torch.int64)
    illegal = torch.zeros((n, stride), dtype=torch.bool, device=dev)
    illegal[:, :cells] = (((me | opp)[:, None] >> bits) & 1) == 1  # occupied cells are never legal
    if A == 65:
        illegal[:, 64] = True  # the pass column: the kernels give a forced pass P = 1 whatever it holds
    equal = torch.stack([3 * z[:, 0], torch.zeros_like(hr[:, 0]), torch.full_like(hr[:, 0], BF16_MAX),
                         torch.full_like(hr[:, 0], -BF16_MAX)], dim=1).gather(1, pick[:, None])
    palette = torch.stack([
        3 * z,
        -(100 + 200 * hr) * u1,
        torch.where(illegal, 30 + 3 * z.abs(), 3 * z),
        equal.expand(n, stride),
        torch.where(u2 < 0.4, sign * BF16_MAX, 3 * z),
        torch.where(u1 < 0.3, sign * 0.0, sub),
    ])
    rows = palette[kind, torch.arange(n, device=dev)]
    s, hv = sign[:, A], hr[:, 0]
    values = torch.stack([2 * z[:, A], s * 0.0, sub[:, A], s * (10 + 990 * hv), s * BF16_MAX], dim=1)
    rows[:, A] = values.gather(1, vkind[:, None])[:, 0]
    rows[:, A + 1:] = BF16_MAX
    return rows.to(torch.bfloat16), kind, vkind


class BoardRowEvaluator:
    """mcts.FusedNetEvaluator's interface with board_rows in place of a net: the row of pending leaf r is
    board_rows(leaf_me[r], leaf_opp[r])"""

    def __init__(self, stride):
        from betazero_b200 import mcts

        self.prior_mode, self.stride = mcts.PRIOR_LOGITS_BF16, int(stride)

    def bind(self, pools):
        self.A, self.R = pools.n_actions, pools.n_rows
        self.out = torch.zeros((max(pools.n_rows, 1), self.stride), dtype=torch.bfloat16, device=pools.device)
        self.value = torch.zeros(1, dtype=torch.float32, device=pools.device)  # unused in this mode
        pools.set_prior_mode(self.prior_mode, self.stride)
        return self.out, self.value

    def __call__(self, pools):
        self.out[: self.R] = board_rows(pools.leaf_me[: self.R], pools.leaf_opp[: self.R], self.A, self.stride)[0]


# ---------------------------------------------------------------------------------------------------------------------
# the node checker
# ---------------------------------------------------------------------------------------------------------------------
def prior_bound(x, p, valid, n):
    """b per edge, such that |P - p| <= b p + 2^-126 (the flush of exp_nonpos: its results below 2^-126 are 0).

    x = l - l_max <= 0 of the edge, p the float64 softmax, n the node's edge count.  A term of the sum is
    exp_nonpos(fl(w - m)): fl(w - m) = x (1 + d), |d| <= 2^-24, which changes e^x by a factor within |x| 2^-24 of 1,
    and exp_nonpos adds its own error (test_gpu_puct_edges.py::test_exp_nonpos_over_every_nonpositive_float):
    e(x) = (1 + 2^-22) 2^dt - 1 + |x| 2^-24, dt = |x| log2(e) (dc + 2^-24 + dc 2^-24).  The n terms (flushed ones off by
    less than 2^-126 each, and the sum s >= 1) sum to S (1 + rho), rho <= sum_j p_j e(x_j) + n 2^-126, and the fp32
    group sum adds at most gamma = (n - 1) 2^-24 / (1 - (n - 1) 2^-24) in any order: s = S (1 +- r), r = rho + gamma +
    rho gamma.  __fdividef(1, s) is within 2 ulp (2^-22), the product w * inv rounds once (2^-24):
    b = (1 + e(x)) (1 + 2^-22) (1 + 2^-24) / (1 - r) - 1."""
    ax = np.where(valid, np.minimum(-x, 1e3), 0.0)  # beyond -1000 the bound is meaningless and p = 0
    dt = ax * LOG2E * (DC + 2.0 ** -24 + DC * 2.0 ** -24)
    e = (1 + 2.0 ** -22) * np.exp2(dt) - 1 + ax * 2.0 ** -24
    gamma = (n - 1) * 2.0 ** -24 / (1 - (n - 1) * 2.0 ** -24)
    rho = np.where(valid, p * e, 0.0).sum(axis=1) + n * 2.0 ** -126
    r = rho + gamma + rho * gamma
    return (1 + e) * (1 + 2.0 ** -22) * (1 + 2.0 ** -24) / (1 - r[:, None]) - 1


def check_nodes(nodes, rows, A, K):
    """Priors and first values of every expanded node (walk_trees) against float64: rows [nodes, >= A + 1] holds each
    node's logits (columns 0..A-1) and pre-tanh value (column A).  Priors within prior_bound of the float64 softmax
    over the node's edges, a forced pass exactly 1; first values by check_search's rule (-tanh, 1e-5 relative +
    4 K 2^-24), values that saturate tanh exactly.  Returns a census of what was checked."""
    valid, act, n = nodes["valid"], nodes["act"].astype(np.int64), nodes["n"]
    lg = np.where(valid, np.take_along_axis(rows, act, axis=1), -np.inf)
    x = lg - lg.max(axis=1, keepdims=True)
    with np.errstate(under="ignore"):
        p = np.exp(x)
    p /= p.sum(axis=1, keepdims=True)
    b = prior_bound(x, p, valid, n)
    P = nodes["P"].astype(np.float64)
    bad = valid & ~(np.abs(P - p) <= b * p + 2.0 ** -126)
    if bad.any():
        i, j = np.argwhere(bad)[0]
        raise AssertionError(f"priors: {int(bad.sum())} edges off, e.g. tree {nodes['tree'][i]}, {n[i]} edges, action "
                             f"{act[i, j]}: logit - max {x[i, j]!r}, P {P[i, j]!r}, float64 {p[i, j]!r}, bound "
                             f"{b[i, j]:.3e} relative")
    near = valid & (x >= -20)
    assert b[near].max() <= 1e-5, b[near].max()  # the north-star's 1e-5 wherever |x| <= 20
    forced = (A == 65) & (n == 1) & (act[:, 0] == 64)
    assert (P[forced, 0] == 1.0).all(), "a forced pass's prior is not 1"

    leaf = (nodes["in_N"] > 0) & ~(valid & (nodes["N"] != 0)).any(axis=1)
    n_in = nodes["in_N"][leaf]
    assert (n_in <= K).all() and (K > 1 or (n_in == 1).all()), np.unique(n_in)
    v = rows[leaf, A]
    t = np.tanh(v)
    W = nodes["in_W"][leaf].astype(np.float64)
    w = W / n_in
    bad = np.abs(w + t) > 1e-5 * np.abs(t) + (0.0 if K == 1 else 4 * K * 2.0 ** -24)
    assert not bad.any(), f"values: {int(bad.sum())} of {len(t)} differ, e.g. W/N {w[bad][:3]} against -tanh {-t[bad][:3]}"
    sat = np.abs(v) >= 10
    assert (W[sat] == -np.sign(v[sat]) * n_in[sat]).all(), "tanhf of |v| >= 10 is not exactly +-1"
    return dict(nodes=len(n), leaves=int(leaf.sum()), leaf=leaf, flushed=int((valid & (P == 0)).sum()),
                saturated=int(sat.sum()), forced_passes=int(forced.sum()),
                illegal_max=int((lg.max(axis=1) < rows[:, :A].max(axis=1)).sum()))


def _node_boards(nodes):
    return (torch.from_numpy(nodes["me"].view(np.int64)).cuda(), torch.from_numpy(nodes["opp"].view(np.int64)).cuda())


def check_row_search(pools, K, stride):
    """check_nodes on a search driven by BoardRowEvaluator: every node's row recomputed from its board.  Returns the
    census with the prior kinds of the nodes and the value kinds of the checked leaves (counts per kind)."""
    nodes = walk_trees(pools)
    rows, kind, vkind = board_rows(*_node_boards(nodes), pools.n_actions, stride)
    rows = rows.double().cpu().numpy()
    census = check_nodes(nodes, rows, pools.n_actions, K)
    kind, vkind = kind.cpu().numpy(), vkind.cpu().numpy()
    leaf = census.pop("leaf")
    census["prior_kinds"] = dict(zip(PRIOR_KINDS, np.bincount(kind, minlength=6).tolist()))
    census["value_kinds"] = dict(zip(VALUE_KINDS, np.bincount(vkind[leaf], minlength=5).tolist()))
    census["equal_20"] = int(((kind == 3) & (nodes["n"] >= 20)).sum())
    return census


# ---------------------------------------------------------------------------------------------------------------------
# roots and searches
# ---------------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _wide_positions(k=32):
    """the k reachable 8x8 positions with the most legal moves (20 .. 23) among 20 000 random playouts"""
    from oracle import pyoracle as po

    me, opp = po.playout_boards(20000, seed=9)
    moves = np.array([bin(int(m)).count("1") for m in po.legal_mask(me, opp)])
    top = np.argsort(-moves, kind="stable")[:k]
    assert moves[top].min() >= 20
    return me[top], opp[top]


def _roots(game, size, B, seed):
    """Reversi: playout positions (midgame, forced passes, finished games), on 8x8 with the 32 widest positions among
    them; tic-tac-toe: 0..5 random moves from the empty board, stopping at a finished game"""
    from betazero_b200 import env, mcts
    from oracle import pyoracle as po

    if game == mcts.GAME_REVERSI:
        me, opp = po.playout_boards(B, seed=seed, size=size)
        if size == 8:
            wm, wo = _wide_positions()
            me[:: B // 32][:32], opp[:: B // 32][:32] = wm, wo
        return env.to_device_u64(me), env.to_device_u64(opp)
    rng = np.random.default_rng(seed)
    me, opp = np.zeros(B, np.uint64), np.zeros(B, np.uint64)
    for i in range(B):
        a, o = 0, 0  # a: the stones of the side to move
        for _ in range(int(rng.integers(0, 6))):
            if po.ttt_terminal(np.array([a]), np.array([o]))[0][0]:
                break
            free = [c for c in range(9) if not ((a | o) >> c) & 1]
            a, o = o, a | (1 << int(rng.choice(free)))
        me[i], opp[i] = a, o
    return env.to_device_u64(me), env.to_device_u64(opp)


def _row_search(game, size, K, group, B, n_sims, stride, fused, seed):
    from betazero_b200 import mcts

    me, opp = _roots(game, size, B, seed)
    pools = mcts.TreePools(B, n_sims, game=game, board_size=size, group_lanes=group, n_leaves=K)
    s = mcts.BatchedMCTS(pools, BoardRowEvaluator(stride), use_graph=False, fused=fused)
    assert not s.one_launch
    s.reset(me, opp)
    s.run(n_sims)
    torch.cuda.synchronize()
    s.check_errors()
    return s


# ---------------------------------------------------------------------------------------------------------------------
# 1-2. the instantiation matrix with board-keyed rows
# ---------------------------------------------------------------------------------------------------------------------
R, T = 0, 1  # mcts.GAME_REVERSI, mcts.GAME_TTT
MATRIX = [  # game, size, K, lanes per tree (0: the dispatch's choice), trees, simulations, stride, fused step
    pytest.param(R, 8, 1, 32, 256, 48, 72, True, id="rev8-K1-32lanes-step"),  # step_kernel<reversi, 32, false>
    pytest.param(R, 8, 1, 32, 256, 32, 80, True, id="rev8-K1-32lanes-stride80"),  # the same, rows 80 bf16 apart
    pytest.param(R, 8, 1, 16, 256, 48, 72, True, id="rev8-K1-16lanes-step"),  # step_kernel<reversi, 16, false>
    pytest.param(R, 8, 1, 8, 256, 48, 72, True, id="rev8-K1-8lanes-step"),  # step_kernel<reversi, 8, false>
    pytest.param(R, 8, 1, 32, 256, 32, 72, False, id="rev8-K1-32lanes-unfused"),  # expand_backup_kernel<reversi, 32, false>
    pytest.param(R, 8, 1, 16, 256, 32, 72, False, id="rev8-K1-16lanes-unfused"),  # expand_backup_kernel<reversi, 16, false>
    pytest.param(R, 8, 1, 8, 256, 32, 72, False, id="rev8-K1-8lanes-unfused"),  # expand_backup_kernel<reversi, 8, false>
    pytest.param(R, 8, 2, 0, 256, 48, 72, True, id="rev8-K2-wave"),  # step_wave_kernel<reversi, 16>
    pytest.param(R, 8, 4, 0, 256, 64, 72, True, id="rev8-K4-wave"),  # step_wave_kernel<reversi, 8>
    pytest.param(R, 8, 3, 0, 256, 48, 72, True, id="rev8-K3-slots-32lanes"),  # step_kernel<reversi, 32, true>
    pytest.param(R, 8, 4, 8, 256, 64, 72, True, id="rev8-K4-slots-8lanes"),  # step_kernel<reversi, 8, true>
    pytest.param(R, 8, 2, 16, 256, 48, 72, True, id="rev8-K2-slots-16lanes"),  # step_kernel<reversi, 16, true>
    pytest.param(R, 8, 1, 0, 8192, 8, 72, True, id="rev8-K1-8192trees-auto16lanes"),  # the dispatch picks 16 lanes
    pytest.param(R, 6, 1, 0, 256, 32, 72, True, id="rev6-K1-32lanes"),
    pytest.param(R, 6, 4, 0, 256, 48, 72, True, id="rev6-K4-wave"),
    pytest.param(R, 4, 1, 0, 256, 24, 72, True, id="rev4-K1-32lanes"),
    pytest.param(R, 4, 4, 0, 256, 32, 72, True, id="rev4-K4-wave"),
    pytest.param(T, 3, 1, 32, 256, 24, 16, True, id="ttt-K1-32lanes"),  # step_kernel<ttt, 32, false>
    pytest.param(T, 3, 1, 16, 256, 24, 16, True, id="ttt-K1-16lanes"),
    pytest.param(T, 3, 1, 8, 256, 24, 16, True, id="ttt-K1-8lanes"),
    pytest.param(T, 3, 2, 32, 256, 24, 16, True, id="ttt-K2-wave"),  # step_wave_kernel<ttt, 16>
    pytest.param(T, 3, 2, 16, 256, 24, 16, True, id="ttt-K2-slots-16lanes"),  # step_kernel<ttt, 16, true>
    pytest.param(T, 3, 2, 8, 256, 24, 16, True, id="ttt-K2-slots-8lanes"),  # step_kernel<ttt, 8, true>
]


@pytest.mark.gpu
@pytest.mark.parametrize("game,size,K,group,B,n_sims,stride,fused", MATRIX)
def test_logits_mode_priors_and_values_in_every_node(game, size, K, group, B, n_sims, stride, fused):
    """Every expanded node of every tree against the float64 softmax and tanh of its board-keyed row; then the census:
    every prior kind among the nodes, every value kind among the checked leaves, flushed priors, saturated values, a
    row maximum on an illegal column, and on 8x8 all-equal rows on nodes with 20+ legal moves."""
    if group == 0 and B >= 8192:
        assert B < 32768  # mcts.cu pool_group: 16 lanes per tree from 8192 to 32767 trees
    s = _row_search(game, size, K, group, B, n_sims, stride, fused, seed=1000 * size + 10 * K + group)
    c = check_row_search(s.pools, K, stride)
    print(f"\n{c}")
    assert c["nodes"] >= B and c["leaves"] >= B // 2, c
    assert min(c["prior_kinds"].values()) > 0 and min(c["value_kinds"].values()) > 0, c
    assert c["flushed"] > 0 and c["saturated"] > 0 and c["illegal_max"] > 0, c
    if game == R and size == 8:
        assert c["equal_20"] > 0, c




@pytest.mark.gpu
def test_the_checker_fails_on_a_prior_or_a_value_off_by_1e_4():
    """The checker has teeth: one root prior, then one first value W (the root edge into a child expanded once),
    multiplied by 1 + 1e-4 in the arena, each make check_row_search fail; restored, it passes again."""
    s = _row_search(R, 8, 1, 32, 256, 48, 72, True, seed=7)
    pools = s.pools
    check_row_search(pools, 1, 72)
    arena = pools.arena.view(pools.n_trees, -1)
    host = arena.cpu().numpy().view(np.uint32)
    meta = pools.root_meta.cpu().numpy().view(np.uint32)
    for t in range(pools.n_trees):
        n, base = int((meta[t] >> 7) & 63), int(meta[t] >> 13) * 8
        edges = host[t, base + 8: base + 8 + 4 * n].reshape(4, n)  # N, W, P, meta of the root's edges
        W, P = edges[1].view(np.float32), edges[2].view(np.float32)
        ok = ((edges[0] == 1) & (((edges[3] >> 7) & 63) > 0) & (np.abs(W) > 1e-3) & (np.abs(W) < 0.999)
              & (P > 1e-3) & (P < 0.999))
        if n > 1 and ok.any():
            e = int(np.flatnonzero(ok)[0])
            break
    else:
        raise AssertionError("no root edge with a child expanded once")
    for word, what in ((base + 8 + 2 * n + e, "priors"), (base + 8 + n + e, "values")):
        old = arena[t, word].clone()
        arena[t, word] = int((host[t, word:word + 1].view(np.float32) * np.float32(1 + 1e-4)).view(np.int32)[0])
        with pytest.raises(AssertionError, match=what):
            check_row_search(pools, 1, 72)
        arena[t, word] = old
    check_row_search(pools, 1, 72)


# ---------------------------------------------------------------------------------------------------------------------
# 3. tic-tac-toe with an exactly representable net
# ---------------------------------------------------------------------------------------------------------------------
def ttt_planes(me, opp):
    """bf16 [n, 9] input of the tic-tac-toe net (the tree kernels' write_planes): +1 the mover's stones, -1 the other's"""
    bit = torch.arange(9, device=me.device)
    return (((me[:, None] >> bit) & 1) - ((opp[:, None] >> bit) & 1)).to(torch.bfloat16)


@pytest.fixture(scope="module")
def ttt_net():
    """exact_net on 9 signed inputs: fc1 rows of 5 weights, logits within about +-15.  The library GEMMs run with fp32
    reductions only (no bf16 split-K reductions), which is what makes an exact net's every partial sum exact."""
    matmul = torch.backends.cuda.matmul
    old = matmul.allow_bf16_reduced_precision_reduction
    matmul.allow_bf16_reduced_precision_reduction = False
    m = exact_net(50, nnz=(5, 16, 16, 16), n_in=9, n_actions=9, device="cuda")
    m.prepare_inference()
    yield m
    matmul.allow_bf16_reduced_precision_reduction = old


def check_ttt_net_search(pools, m, K):
    """check_nodes with the float64 net: the library GEMMs on the nodes' planes equal it bit for bit (the premise),
    and the tree's priors and values are its softmax and tanh"""
    nodes = walk_trees(pools)
    x = ttt_planes(*_node_boards(nodes))
    check_exact(m, x)
    ref = reference_forward(x, m)
    assert torch.equal(m.forward_raw(x)[:, :10].double(), ref), "the library GEMMs are not the float64 net"
    return check_nodes(nodes, ref.cpu().numpy(), 9, K)


@pytest.mark.gpu
@pytest.mark.parametrize("group", [8, 16, 32])
@pytest.mark.parametrize("K", [1, 2])
def test_ttt_search_with_an_exact_net(ttt_net, K, group):
    """FusedNetEvaluator on the tic-tac-toe net (library GEMMs, rows 16 bf16 apart): every node of 256 trees"""
    from betazero_b200 import mcts

    me, opp = _roots(T, 3, 256, seed=K * 100 + group)
    ev = mcts.FusedNetEvaluator(ttt_net)
    s = mcts.BatchedMCTS(mcts.TreePools(256, 32, game=mcts.GAME_TTT, group_lanes=group, n_leaves=K), ev, use_graph=False)
    assert ev.stride == 16 and ev.own_launches == 0
    s.search(me, opp, 32)
    torch.cuda.synchronize()
    c = check_ttt_net_search(s.pools, ttt_net, K)
    assert c["nodes"] >= 256 and c["leaves"] >= 128, c


@pytest.mark.gpu
def test_ttt_player_with_an_exact_net_in_the_reference_loop(ttt_net):
    """BASELINE config 1 with a net: TicTacToeMCTSPlayer(net=...) for both sides in the reference's headless loop, the
    tree of every move checked"""
    from helpers import play_ttt_headless

    from betazero_b200 import mcts
    from betazero_b200.boards import TicTacToeBoard
    from betazero_b200.players import TicTacToeMCTSPlayer

    checked = []

    class Checked(TicTacToeMCTSPlayer):
        def get_move(self, board):
            mv = super().get_move(board)
            assert isinstance(self.search.evaluator, mcts.FusedNetEvaluator)
            checked.append(check_ttt_net_search(self.pools, ttt_net, 1))
            return mv

    positions, _ = play_ttt_headless(TicTacToeBoard, Checked(1, net=ttt_net, n_sims=100), Checked(-1, net=ttt_net, n_sims=100))
    assert len(checked) == len(positions) - 1 >= 5
    assert sum(c["nodes"] for c in checked) >= 100


# ---------------------------------------------------------------------------------------------------------------------
# 4. the one-launch search at the edges of the range
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def scaled_nets():
    """test_net_exact's search net (seed 21) with the head's weights and biases times 2^s: still exact, the grid unit
    scales with them"""
    nets = {}
    for scale in (40, -60):
        m = exact_net(21, shifts=(0, 0, 0, 12 - scale), device="cuda")
        m.prepare_inference()
        nets[scale] = m
    return nets


@pytest.mark.gpu
@pytest.mark.parametrize("scale", [40, -60])
@pytest.mark.parametrize("K", [1, 2, 4])
@pytest.mark.parametrize("B,n_sims", [(57, 32), (4145, 16)])
def test_one_launch_search_with_a_scaled_head(scaled_nets, scale, K, B, n_sims):
    """bz_mcts_search_fused with the head scaled by 2^40 (logit spreads of about 2^40: every prior but the maxima
    flushes to 0, tanh is exactly +-1) and by 2^-60 (logits and values near 2^-60, normal floats): every node against
    the float64 net (check_search), and the same trees as the per-iteration kernels"""
    from test_net_exact import planes_of

    m = scaled_nets[scale]
    me, opp = _net_roots(B, "playout", 8, seed=B + K + abs(scale))
    a = _fused_search(m, me, opp, n_sims, K, 8, True)
    nodes, leaves = check_search(a.pools, [m], np.zeros(B, np.int64), K)
    assert nodes >= B // 2 and leaves >= B // 4, (nodes, leaves)
    _same_trees(a, _fused_search(m, me, opp, n_sims, K, 8, False))
    nd = walk_trees(a.pools)
    ref = reference_forward(planes_of(*_node_boards(nd)), m).abs()
    assert ref.max() < BF16_MAX
    flushed = int((nd["valid"] & (nd["P"] == 0)).sum())
    if scale > 0:
        assert flushed > 0 and bool((torch.tanh(ref[:, 65]).float() == 1).any()), flushed
    else:
        assert flushed == 0 and ref.max() < 2.0 ** -40 and ref[ref > 0].min() >= 2.0 ** -126
