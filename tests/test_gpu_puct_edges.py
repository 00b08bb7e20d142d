"""The PUCT score where the straight-line arithmetic hands over to the exact form.

Every score in the tree kernels is computed by `puct_score_straight` (betazero_b200/csrc/puct.cuh): a division by a
visit count without the range check of `__fdiv_rn`, and sqrt(n) from a table.  A warp vote falls back to the exact
`puct_score` when an operand lies outside [2^-100, 2^100] or a node has 65 536 visits or more.  The fallback is written
out three times in mcts.cu (score_pass for 16 and 32 lanes, the two-edge pass for 8 lanes, the root choices of wave
mode), and nothing else in the suite sends priors, values or W that far out.

1. Extreme priors and values in lockstep with the C oracle, in every kernel family, with a walk of the GPU trees that
   proves the fallback was taken.
2. The primitives over their domain, through a harness (tests/puct_harness.cu) built with the library's nvcc flags.
3. The one-launch search with a net peaked enough that priors fall below 2^-106 or flush to 0, against the per-iteration
   kernels, node block by node block.
"""
import ctypes
import fcntl
import hashlib
import math
import os
import subprocess

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from test_gpu_one_launch import _same_trees  # noqa: E402
from test_net_exact import _roots as _net_roots  # noqa: E402
from test_net_exact import walk_trees  # noqa: E402

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HARNESS_SRC = os.path.join(ROOT, "tests", "puct_harness.cu")
HEADER = os.path.join(ROOT, "betazero_b200", "csrc", "puct.cuh")
HARNESS_DIR = os.path.join(ROOT, "build", "puct_harness")
HARNESS_SO = os.path.join(HARNESS_DIR, "libpuct_harness.so")

LO, HI = 2.0 ** -100, 2.0 ** 100  # the straight-line division's range (fdiv_by_count)
P = ctypes.c_void_p


# ---------------------------------------------------------------------------------------------------------------------
# the harness: built on first use like oracle/pyendgame.py's library (content hash, lock, atomic rename)
# ---------------------------------------------------------------------------------------------------------------------
def _harness_flags():
    from betazero_b200 import build as bz_build

    return [f for f in bz_build.NVCC_FLAGS if f != "-lineinfo"]


def _harness_hash():
    h = hashlib.sha256(" ".join(_harness_flags()).encode())
    for path in (HARNESS_SRC, HEADER):
        with open(path, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def _build_harness():
    from betazero_b200 import build as bz_build

    stamp = HARNESS_SO + ".srchash"

    def stale():
        try:
            return not os.path.exists(HARNESS_SO) or open(stamp).read().strip() != _harness_hash()
        except OSError:
            return True

    if not stale():
        return HARNESS_SO
    os.makedirs(HARNESS_DIR, exist_ok=True)
    with open(HARNESS_SO + ".lock", "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if stale():
                tmp = f"{HARNESS_SO}.tmp.{os.getpid()}"
                subprocess.check_call([bz_build._nvcc(), *_harness_flags(), "-o", tmp, HARNESS_SRC])
                os.replace(tmp, HARNESS_SO)
                with open(stamp + ".tmp", "w") as f:
                    f.write(_harness_hash())
                os.replace(stamp + ".tmp", stamp)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return HARNESS_SO


@pytest.fixture(scope="module")
def harness():
    L = ctypes.CDLL(_build_harness())
    L.puct_fdiv_sweep.argtypes = [ctypes.c_uint, ctypes.c_uint, ctypes.c_int, ctypes.c_uint, P, P]
    L.puct_order_key_sweep.argtypes = [P, P]
    L.puct_exp_sweep.argtypes = [ctypes.c_double, ctypes.c_double, P, P, P]
    L.puct_fdiv_map.argtypes = [P, P, P, P, ctypes.c_int]
    L.puct_score_map.argtypes = [P, P, P, P, ctypes.c_float, P, P, P, ctypes.c_int]
    L.puct_sqrt_map.argtypes = [P, P, P, ctypes.c_int]
    assert L.puct_fill_sqrt_table() == 0
    return L


def _ptr(a):
    return a.ctypes.data_as(P)


def _sweep(fn, *args, maxes=False):
    count = np.zeros(16, np.uint64)
    rec = np.zeros(1 + 4 * 8, np.uint32)
    out = [count, rec]
    extra = []
    if maxes:
        m = np.zeros(4, np.float64)
        extra, out = [_ptr(m)], out + [m]
    assert fn(*args, _ptr(count), _ptr(rec), *extra) == 0
    return out


def _records(rec):
    n = min(int(rec[0]), 8)
    return [tuple(f"{int(x):#010x}" for x in rec[1 + 4 * i: 5 + 4 * i]) for i in range(n)]


# ---------------------------------------------------------------------------------------------------------------------
# 2. the primitives over their domain
# ---------------------------------------------------------------------------------------------------------------------
def test_fdiv_by_count_is_fdiv_rn_for_every_divisor(harness):
    """Every divisor in [1, 2^24] with 64 numerators each (tests/puct_harness.cu, sweep_numerator): +-0, the range ends
    2^-100 and 2^100 with their float neighbours inside and outside, 1, FLT_MAX, the smallest normal, denormals, inf,
    NaN, d and d + 1 ulp, random mantissas at exponents over [-100, 100) and over every normal exponent, and numerators
    whose quotient lies within 1/d of an ulp from a rounding midpoint.  Inside the range the straight-line quotient is
    __fdiv_rn bit for bit; a zero numerator gives a zero that leaves u >= +0 unchanged; `bad` is set exactly for
    nonzero numerators outside the range, inf and NaN."""
    n_div, per = 1 << 24, 64
    count, rec = _sweep(harness.puct_fdiv_sweep, 1, n_div, per, 7)
    assert int(count[0]) == n_div * per
    assert int(count[5]) == 0, f"`bad` wrong in {int(count[5])} cases: {_records(rec)}"
    assert int(count[2]) == 0, f"{int(count[2])} in-range quotients differ from __fdiv_rn: {_records(rec)}"
    assert int(count[4]) == 0, f"{int(count[4])} zero numerators break the sign claim: {_records(rec)}"
    assert int(count[3]) == 2 * n_div
    assert int(count[8]) > n_div, "too few numerators next to a rounding midpoint"
    assert int(count[9]) == 0
    print(f"\nfdiv_by_count: {int(count[1])} in-range quotients equal __fdiv_rn ({int(count[8])} within 1/d ulp of a "
          f"midpoint); outside the range the straight result differs from __fdiv_rn in {int(count[7])} of "
          f"{int(count[6])} cases ({int(count[7]) / max(int(count[6]), 1):.1%}), for finite numerators in {int(count[10])} of "
          f"{int(count[11])}: the work the guard does")


def _numerators(rng, n):
    """float32 numerators: in range (random mantissa, exponent in [-100, 100]), the ends and their neighbours, zeros,
    denormals, out of range on both sides, inf and NaN"""
    kind = rng.integers(0, 8, n)
    mant = rng.integers(0, 1 << 23, n, dtype=np.uint32)
    sign = rng.integers(0, 2, n, dtype=np.uint32) << np.uint32(31)
    exp_in = rng.integers(27, 228, n, dtype=np.uint32)  # biased: 2^-100 .. 2^100 (the top one is only 2^100 itself)
    bits = np.where(exp_in == 227, np.uint32(227 << 23), (exp_in << np.uint32(23)) | mant)
    ends = np.array([0x0D800000, 0x0D800001, 0x0D7FFFFF, 0x71800000, 0x717FFFFF, 0x71800001], np.uint32)
    exp_out = np.where(rng.random(n) < 0.5, rng.integers(1, 27, n), rng.integers(228, 255, n)).astype(np.uint32)
    specials = np.array([0, 0x7F800000, 0x7FC00000, 0x7F7FFFFF, 0x00800000], np.uint32)
    bits = np.select([kind < 4, kind == 4, kind == 5, kind == 6],
                     [bits, ends[rng.integers(0, 6, n)], mant | 1, (exp_out << np.uint32(23)) | mant],
                     specials[rng.integers(0, 5, n)]).astype(np.uint32)
    return (bits | sign).view(np.float32)


def test_fdiv_by_count_sampled_against_float64(harness):
    """1 M sampled (numerator, divisor) pairs against numpy: float64 division rounded to float32 is the correctly
    rounded float32 quotient (53 >= 2 * 24 + 2 bits: the double rounding is innocuous), so in range the straight-line
    quotient must equal it bit for bit, independently of __fdiv_rn."""
    rng = np.random.default_rng(11)
    n = 1 << 20
    num = _numerators(rng, n)
    den = np.where(rng.random(n) < 0.5, rng.integers(1, 1025, n), rng.integers(1, (1 << 24) + 1, n)).astype(np.float32)
    q = np.empty(n, np.float32)
    bad = np.empty(n, np.uint8)
    assert harness.puct_fdiv_map(_ptr(num), _ptr(den), _ptr(q), _ptr(bad), n) == 0
    a = num.view(np.uint32) & np.uint32(0x7FFFFFFF)
    inside = (a >= 0x0D800000) & (a <= 0x71800000)
    zero = a == 0
    assert np.array_equal(bad.astype(bool), ~zero & ~inside)
    with np.errstate(all="ignore"):
        want = (num.astype(np.float64) / den.astype(np.float64)).astype(np.float32)
    sel = inside & ~zero
    diff = np.flatnonzero(q[sel].view(np.uint32) != want[sel].view(np.uint32))
    assert len(diff) == 0, [(float(num[sel][i]), float(den[sel][i]), float(q[sel][i]), float(want[sel][i])) for i in diff[:5]]
    assert (q[zero] == 0).all() and ((q[zero] + np.float32(0)).view(np.uint32) == 0).all()
    assert sel.sum() > n // 2 and zero.sum() > 1000 and (~zero & ~inside).sum() > n // 8


def _score_operands(rng, n):
    N = np.select([rng.random(n) < 0.6, rng.random(n) < 0.5],
                  [rng.integers(0, 64, n), rng.integers(0, 65536, n)], rng.integers(0, 1 << 24, n)).astype(np.int32)
    W = np.where(rng.random(n) < 0.3, rng.uniform(-1, 1, n) * N, 0).astype(np.float32)
    k = rng.integers(0, 6, n)
    tiny = np.ldexp(rng.uniform(0.5, 1, n), -rng.integers(90, 150, n))
    huge = np.ldexp(rng.uniform(0.5, 1, n), rng.integers(90, 120, n))
    sgn = np.where(rng.random(n) < 0.5, -1.0, 1.0)
    W = np.select([k == 0, k == 1, k == 2, k == 3], [W, sgn * tiny, sgn * huge, np.where(rng.random(n) < 0.5, 0.0, -0.0)],
                  rng.uniform(-2, 2, n)).astype(np.float32)
    Pk = rng.integers(0, 5, n)
    Pr = np.select([Pk == 0, Pk == 1, Pk == 2, Pk == 3],
                   [rng.random(n), np.ldexp(rng.uniform(0.5, 1, n), -rng.integers(1, 150, n)), 0.0 * rng.random(n),
                    -0.0 * np.ones(n)], np.ldexp(rng.uniform(0.5, 1, n), -rng.integers(100, 130, n))).astype(np.float32)
    n_node = np.where(rng.random(n) < 0.5, rng.integers(1, 65536, n), rng.integers(1, 1 << 24, n))
    sq = np.sqrt(n_node.astype(np.float64)).astype(np.float32)
    return N, W, Pr, sq


def test_straight_score_equals_puct_score_when_the_guard_stays_clear(harness):
    """puct_score_straight against puct_score on 1 M operand sets with extreme W and P: equal as floats (-0 == +0)
    whenever `bad` stays clear; and puct_score itself against its float32 restatement in numpy (IEEE, denormals kept)."""
    rng = np.random.default_rng(12)
    n = 1 << 20
    N, W, Pr, sq = _score_operands(rng, n)
    for c in (1.25, 2.0):
        st, ex = np.empty(n, np.float32), np.empty(n, np.float32)
        bad = np.empty(n, np.uint8)
        assert harness.puct_score_map(_ptr(N), _ptr(W), _ptr(Pr), _ptr(sq), c, _ptr(st), _ptr(bad), _ptr(ex), n) == 0
        clear = bad == 0
        diff = np.flatnonzero(clear & (st != ex))
        assert len(diff) == 0, [(int(N[i]), float(W[i]), float(Pr[i]), float(sq[i]), float(st[i]), float(ex[i]))
                                for i in diff[:5]]
        assert 0.2 * n < clear.sum() < 0.9 * n, clear.sum()
        f = np.float32
        with np.errstate(all="ignore"):
            q = np.where(N > 0, W / np.maximum(N, 1).astype(np.float32), f(0)).astype(np.float32)
            u = (((f(c) * Pr) * sq) / (N + 1).astype(np.float32)).astype(np.float32)
            ref = (q + u).astype(np.float32)
        wrong = np.flatnonzero(ex.view(np.uint32) != ref.view(np.uint32))
        assert len(wrong) == 0, [(int(N[i]), float(W[i]), float(Pr[i]), float(ex[i]), float(ref[i])) for i in wrong[:5]]


def test_sqrt_table_and_its_accessors(harness):
    """g_sqrt_tab[n] (read through both accessors) is the correctly rounded sqrt for every n < 65536; sqrt_of_count is
    correct at 65536, at 2^24 and on a sample between; sqrt_of_small_count clamps to the last entry."""
    rng = np.random.default_rng(13)
    big = np.concatenate([[65536, 65537, (1 << 24) - 1, 1 << 24], rng.integers(65536, (1 << 24) + 1, 100000)])
    n = np.concatenate([np.arange(65536), big]).astype(np.int32)
    small, full = np.empty(len(n), np.float32), np.empty(len(n), np.float32)
    assert harness.puct_sqrt_map(_ptr(n), _ptr(small), _ptr(full), len(n)) == 0
    want = np.sqrt(n.astype(np.float32).astype(np.float64)).astype(np.float32)  # 53 >= 2 * 24 + 2: correctly rounded
    assert np.array_equal(full.view(np.uint32), want.view(np.uint32))
    assert np.array_equal(small[:65536].view(np.uint32), want[:65536].view(np.uint32))
    assert (small[65536:].view(np.uint32) == want[65535].view(np.uint32)).all()


def test_order_key_is_strictly_monotone_over_every_float(harness):
    """all 2^32 bit patterns but NaN, each against its successor in the float order: strictly increasing keys, the same
    key for -0 and +0, and no key 0 (the lanes that score no edge use 0)"""
    count, rec = _sweep(harness.puct_order_key_sweep)
    non_nan = (1 << 32) - 2 * ((1 << 23) - 1)
    assert int(count[0]) == non_nan - 1
    assert int(count[1]) == 0, f"{int(count[1])} pairs out of order: {_records(rec)}"
    assert int(count[2]) == 0, f"{int(count[2])} zero keys: {_records(rec)}"


def test_exp_nonpos_over_every_nonpositive_float(harness):
    """exp_nonpos(x) = ex2.approx.ftz(fl(x * fl(log2 e))) for every float x <= 0 against exp((double) x).

    The bound: with t = fl(x * L'), L' = fl(log2 e) = log2 e (1 + dc), t = x log2 e (1 + dc)(1 + dm), |dm| <= 2^-24, so
    |t - x log2 e| <= |x| log2 e (|dc| + 2^-24 + |dc| 2^-24) =: dt and 2^t / e^x is within a factor 2^(+-dt) of 1.
    ex2.approx.f32 has a relative error of at most 2^-22 (PTX ISA), so |y - e^x| / e^x <= (1 + 2^-22) 2^dt - 1 --
    about 2^-22 + |x| 2^-24 near 0, 1e-5 near x = -87.  Results below 2^-126 are flushed: every nonzero result is
    normal, a 0 is only allowed where e^x (1 + bound) can fall below 2^-126, and exp_nonpos(+-0) == 1."""
    dc = abs(float(np.float32(1.4426950408889634)) - 1.4426950408889634) / 1.4426950408889634 + 2.0 ** -52
    err2 = 2.0 ** -22
    count, rec, maxes = _sweep(harness.puct_exp_sweep, err2, dc, maxes=True)
    assert int(count[0]) == 0x7F800002  # -0 .. -inf, and +0
    names = {1: "over the bound", 2: "denormal results", 3: "flushed although above 2^-126",
             4: "not flushed although below 2^-126", 5: "exp_nonpos(+-0) != 1"}
    for k, what in names.items():
        assert int(count[k]) == 0, f"{int(count[k])} {what}: {_records(rec)}"
    assert int(count[6]) > 1 << 30
    print(f"\nexp_nonpos: max relative error {maxes[0]:.3e} (ex2.approx alone {maxes[1]:.3e} = 2^{math.log2(maxes[1]):.2f}); "
          f"largest error / bound {maxes[2]:.3f}")


# ---------------------------------------------------------------------------------------------------------------------
# 1. extreme operands in lockstep with the C oracle
# ---------------------------------------------------------------------------------------------------------------------
def _extreme_weights(rng, rows, A):
    """each row: ordinary weights, m 2^-e with e in [0, 160] (normals, the band below 2^-100, denormals, underflow to 0),
    one dominant weight over weights near 2^-120, or all zeros (+0 and -0: the uniform rule); exact zeros and -0.0
    sprinkled over the others"""
    kind = rng.integers(0, 10, rows)[:, None]
    ordinary = rng.random((rows, A)) ** 4
    scaled = np.ldexp(rng.uniform(0.5, 1, (rows, A)), -rng.integers(0, 161, (rows, A)))
    dominant = np.ldexp(rng.uniform(0.5, 2, (rows, A)), -120)
    dominant[np.arange(rows), rng.integers(0, A, rows)] = 1.0
    w = np.select([kind < 3, kind < 6, kind < 9], [ordinary, scaled, dominant], 0.0).astype(np.float32)
    z = rng.random((rows, A))
    w[z < 0.1] = 0.0
    w[(z > 0.95) | ((kind == 9) & (z < 0.5))] = -0.0
    return w


def _extreme_values(rng, rows):
    """ordinary, +-2^-k (k <= 149: denormals), +-0, +-1/2 and +-1/4 (sums that cancel W exactly), and a few magnitudes
    up to 2^110 (|W| beyond 2^100 without overflow)"""
    kind = rng.random(rows)
    sgn = np.where(rng.random(rows) < 0.5, -1.0, 1.0)
    v = np.select([kind < 0.3, kind < 0.55, kind < 0.65, kind < 0.95],
                  [rng.uniform(-1, 1, rows), sgn * np.ldexp(1.0, -rng.integers(1, 150, rows)), sgn * 0.0,
                   sgn * np.ldexp(1.0, -rng.integers(1, 3, rows))],
                  sgn * np.ldexp(rng.uniform(0.5, 1, rows), rng.integers(90, 111, rows)))
    return v.astype(np.float32)


def _out_of_range(x):
    a = np.abs(x.astype(np.float64))
    return (a != 0) & ((a < LO) | (a > HI))


def _fallback_nodes(pools, c, sims):
    """from the final trees: per node, whether an edge's u numerator fl(fl(c P) sqrt(n)) or its W is nonzero and
    outside [2^-100, 2^100], on nodes with at least 2 visits (roots: the trees' iteration counts)"""
    nd = walk_trees(pools)
    root = nd["in_N"] < 0
    n_node = np.where(root, sims[nd["tree"]], nd["in_N"])
    sq = np.sqrt(n_node.astype(np.float64)).astype(np.float32)[:, None]
    with np.errstate(all="ignore"):
        unum = (np.float32(c) * nd["P"]) * sq
    valid = nd["valid"] & (n_node >= 2)[:, None]
    u_out = (valid & _out_of_range(unum)).any(1)
    w_out = (valid & _out_of_range(nd["W"])).any(1)
    wide = (nd["n"] > 8) & (valid & (_out_of_range(unum) | _out_of_range(nd["W"])) & (np.arange(33) >= 8)[None, :]).any(1)
    return dict(root=root, u=u_out, w=w_out, wide=wide)


def _lockstep(game, size, K, group, B, iters, seed, c=2.0):
    """the same extreme (w, v) to the GPU trees and the C trees every iteration; leaves, statuses and path lengths of
    every slot, then the root statistics, bit for bit.  Returns the fallback census of the GPU trees."""
    from betazero_b200 import env, mcts
    from oracle import pyoracle as po

    if game == mcts.GAME_TTT:
        x = np.array([0, 0b000010000, 0b100000001, 0], dtype=np.uint64)
        o = np.array([0, 0b000000001, 0b000010010, 0], dtype=np.uint64)
        me_h, opp_h = np.resize(x, B), np.resize(o, B)
    else:
        me_h, opp_h = po.playout_boards(B, seed=seed, size=size)
    A = 9 if game == mcts.GAME_TTT else 65
    pools = mcts.TreePools(B, iters * K, game=game, board_size=size, c_puct=c, group_lanes=group, n_leaves=K)
    s = mcts.BatchedMCTS(pools, None, use_graph=False)
    s.reset(env.to_device_u64(me_h), env.to_device_u64(opp_h))
    trees = [po.OracleTree(game, size, c) for _ in range(B)]
    for t, m, o in zip(trees, me_h, opp_h):
        t.reset_wire(m, o)
    rng = np.random.default_rng(seed)
    s.select()
    for it in range(iters):
        lm, lo = env.to_host_u64(pools.leaf_me), env.to_host_u64(pools.leaf_opp)
        st = pools.leaf_status.cpu().numpy()
        plen = pools.path_len.cpu().numpy()
        w = _extreme_weights(rng, K * B, A)
        v = _extreme_values(rng, K * B)
        for i, t in enumerate(trees):
            for j in range(K):
                r = j * B + i
                got = (int(st[r]), int(lm[r]), int(lo[r]), int(plen[r]))
                assert (t.select() if K == 1 else t.select_vl(j)) == got, (it, i, j)
            for j in range(K):
                r = j * B + i
                if K == 1:
                    t.expand_backup(w[r], v[r])
                else:
                    t.expand_backup_vl(j, w[r], v[r])
        s.prior_w.copy_(torch.from_numpy(w))
        s.value.copy_(torch.from_numpy(v))
        if it + 1 < iters:
            s.step()
        else:
            s.expand_backup()
    cnt, _, _ = (x.cpu().numpy() for x in s.root_policy())
    _, W, Pr = (x.cpu().numpy() for x in s.root_edges())
    for i, t in enumerate(trees):
        rc, rw, rp = t.root_stats()
        assert np.array_equal(cnt[i], rc) and np.array_equal(W[i], rw) and np.array_equal(Pr[i], rp), i
    s.check_errors()
    return _fallback_nodes(pools, c, pools.sim_count.cpu().numpy())


LOCKSTEP = [  # game, size, K, lanes per tree, trees, iterations, seed: which kernels (mcts.cu dispatch) run
    pytest.param(0, 8, 1, 32, 64, 60, 1, id="K1-32lanes"),  # select/step_kernel<reversi, 32, false>: score_pass + redux
    pytest.param(0, 8, 1, 16, 64, 60, 2, id="K1-16lanes"),  # <reversi, 16, false>: score_pass, butterfly on floats
    pytest.param(0, 8, 1, 8, 64, 60, 3, id="K1-8lanes"),  # <reversi, 8, false>: the two-edge pass, `wide` (> 8 edges)
    pytest.param(0, 8, 2, 0, 48, 40, 4, id="K2-wave"),  # select/step_wave_kernel<reversi, 16>: root choices + 16 lanes
    pytest.param(0, 8, 4, 0, 48, 30, 5, id="K4-wave"),  # select/step_wave_kernel<reversi, 8>: root choices + 8 lanes
    pytest.param(0, 8, 3, 0, 48, 30, 6, id="K3-slots"),  # select/step_kernel<reversi, 32, true>: slots one after the other
    pytest.param(1, 3, 1, 8, 64, 50, 7, id="ttt-K1-8lanes"),  # <ttt, 8, false>: the empty board's 9 edges take `wide`
]


@pytest.mark.parametrize("game,size,K,group,B,iters,seed", LOCKSTEP)
def test_extreme_priors_and_values_in_lockstep_with_the_oracle(game, size, K, group, B, iters, seed):
    """Priors m 2^-e (e <= 160), one dominant weight over 2^-120, zeros, -0, all-zero rows; values 2^-k (k <= 149),
    +-0, cancelling halves and quarters, magnitudes up to 2^110.  The trees must be the oracle's; then the walk of the
    GPU trees must find nodes with 2+ visits whose scores took the fallback through an out-of-range u numerator and
    through an out-of-range W (and, with 8 lanes, on an edge of the second set; in wave mode, at the roots)."""
    census = _lockstep(game, size, K, group, B, iters, seed)
    u, w, root = census["u"], census["w"], census["root"]
    msg = {k: int(v.sum()) for k, v in census.items()}
    assert u.sum() >= B // 4 and w.sum() >= B // 8, msg
    if group == 8:
        assert census["wide"].sum() >= 4, msg
    if K in (2, 4):
        assert (root & (u | w)).sum() >= B // 4, msg


@pytest.mark.parametrize("group", [32, 16])
def test_root_counts_beyond_the_sqrt_table_with_16_and_32_lanes(group):
    """score_pass (16 and 32 lanes per tree) at roots with more than 65536 visits, where the vote must take sqrt(n)
    from sqrt_of_count rather than the clamped table: 32 trees on 4x4 boards, 70000 iterations, bit for bit against the
    oracle (test_gpu_mcts.py covers the default width with 6 trees)."""
    from betazero_b200 import env, mcts
    from oracle import pyoracle as po

    B, S, c = 32, 70000, 2.0
    me_h, opp_h = po.playout_boards(B, seed=17, size=4)
    me_h[0], opp_h[0] = po.grid_to_wire(po.OracleReversiBoard(size=4).board, 1)
    pools = mcts.TreePools(B, S, board_size=4, c_puct=c, group_lanes=group, arena_units=400000)
    s = mcts.BatchedMCTS(pools, mcts.HashEvaluator(3))
    cnt, _, _ = s.search(env.to_device_u64(me_h), env.to_device_u64(opp_h), S)
    r_cnt, r_W, r_P, _ = po.search_hash(me_h, opp_h, S, po.GAME_REVERSI, 4, c, 3)
    assert (r_cnt.sum(1) > 65536).sum() >= B // 2
    assert np.array_equal(cnt.cpu().numpy(), r_cnt)
    _, W, Pr = (x.cpu().numpy() for x in s.root_edges())
    assert np.array_equal(W, r_W) and np.array_equal(Pr, r_P)


# ---------------------------------------------------------------------------------------------------------------------
# 3. the one-launch search with a peaked net
# ---------------------------------------------------------------------------------------------------------------------
def _peaked_net(seed):
    """make_net("mlp") with the policy rows scaled by 512 (even actions) and 1024 (odd actions), powers of two so the
    bf16 weights scale exactly: the untrained net's logit spreads of 0.1 .. 0.2 between legal moves become 50 .. 200, so
    priors land below 2^-106 (spreads past 73.5: the fallback) and below 2^-126 (past 87.3: flushed to 0)"""
    from betazero_b200 import net

    m = net.make_net("mlp", seed=seed)
    scale = torch.where(torch.arange(m.policy.out_features, device="cuda") % 2 == 0, 512.0, 1024.0).to(m.policy.weight.dtype)
    with torch.no_grad():
        m.policy.weight.mul_(scale[:, None])
        m.policy.bias.mul_(scale)
    return m


def _fused_search(model, me, opp, n_sims, K, size, one_launch):
    from betazero_b200 import mcts

    s = mcts.BatchedMCTS(mcts.TreePools(me.numel(), n_sims, board_size=size, n_leaves=K), mcts.FusedNetEvaluator(model),
                         use_graph=False, one_launch=one_launch)
    assert s.one_launch is one_launch
    s.pools.arena.zero_()  # the padding words at the end of a node block are never written: make them comparable
    s.reset(me, opp)
    s.run(n_sims)
    torch.cuda.synchronize()
    s.check_errors()
    return s


@pytest.mark.parametrize("K", [1, 2, 4])
@pytest.mark.parametrize("B,size,n_sims", [(300, 8, 64), (4145, 8, 16), (300, 6, 64), (4145, 6, 16)])
def test_one_launch_search_with_a_peaked_net_builds_the_same_trees(K, B, size, n_sims):
    """bz_mcts_search_fused against the per-iteration kernels with the bf16 logits of a peaked net (4145 trees: two
    launches), every node block bit for bit; the walk must find priors in (0, 2^-106] on nodes visited twice or more
    (their scores take the fallback) and priors flushed to exactly 0."""
    model = _peaked_net(K * 10 + size)
    me, opp = _net_roots(B, "playout", size, seed=B + K)
    a = _fused_search(model, me, opp, n_sims, K, size, True)
    b = _fused_search(model, me, opp, n_sims, K, size, False)
    _same_trees(a, b)
    nd = walk_trees(a.pools)
    sims = a.pools.sim_count.cpu().numpy()
    n_node = np.where(nd["in_N"] < 0, sims[nd["tree"]], nd["in_N"])
    visited = nd["valid"] & (n_node >= 2)[:, None]
    tiny = (visited & (nd["P"] > 0) & (nd["P"] <= 2.0 ** -106)).any(1).sum()
    flushed = (nd["valid"] & (nd["P"] == 0)).any(1).sum()
    assert tiny >= B // 10 and flushed >= B // 10, (int(tiny), int(flushed))
