"""Batched net-versus-net matches: thousands of games between two nets on one GPU, every move searched with the
one-launch kernel -- the evaluation the AlphaZero loop needs after an iteration (did the new net get stronger?).

Games 2i and 2i+1 form pair i: both start with the same ``opening_plies`` uniformly random legal moves (Philox keyed by
seed, pair id, ply), then net A plays X in game 2i and net B plays X in game 2i+1.  Each ply:

    bz_match_layout (A's movers -> trees [0, nA), B's from the next multiple of 56)
    -> bz_mcts_reset -> bz_mcts_search_fused_two_nets (each CTA pair loads its own net) -> bz_match_advance

A move is the most visited root action, lowest action id on ties -- ``MCTSPlayer.get_move`` with the same net, ``n_sims``,
``n_leaves`` and ``c_puct``, so every game can be replayed move for move with the sequential players of ``arena.py``.
Pairs are the independent unit of the score's interval: the two games of a pair share their opening.

    python -m betazero_b200.match --a A.pt --b B.pt --games 4088 --sims 800 --leaves 4
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import time

import torch

from . import _lib
from ._lib import BzMatchState, BzTreePools
from .mcts import PRIOR_LOGITS_BF16, TreePools

TREES_PER_PAIR = 56      # a CTA pair of the one-launch kernel: the unit that loads one net
MAX_PLIES = 128          # BZ_MATCH_MAX_PLIES
RUNNING = 2              # BZ_MATCH_RUNNING
Z95 = 1.959963984540054  # two-sided 95 % normal quantile


def elo(score: float) -> float:
    """Elo difference of an expected score in [0, 1] (logistic model); +-inf at 1 and 0."""
    if score >= 1.0:
        return math.inf
    if score <= 0.0:
        return -math.inf
    return -400.0 * math.log10(1.0 / score - 1.0)


def elo_summary(pair_scores) -> dict:
    """Score, Elo and a 95 % interval from the mean score of each pair (its two games' mean: 0, 1/4, 1/2, 3/4 or 1).
    The interval is the normal interval of the mean pair score (standard error with n - 1), mapped through ``elo``."""
    xs = [float(x) for x in pair_scores]
    n = len(xs)
    if n == 0:
        return {"score": math.nan, "elo": math.nan, "elo_ci": [math.nan, math.nan], "score_se": math.nan, "pairs": 0}
    mean = sum(xs) / n
    se = math.sqrt(sum((x - mean) ** 2 for x in xs) / (n - 1) / n) if n > 1 else 0.0
    lo, hi = mean - Z95 * se, mean + Z95 * se
    return {"score": mean, "elo": elo(mean), "elo_ci": [elo(lo), elo(hi)], "score_se": se, "pairs": n}


def check_net(net) -> None:
    """The one-launch kernel covers the bf16 128-256-256-256-(65+1) MLP only; there is no other path."""
    from .net import PolicyValueMLP

    ok = (isinstance(net, PolicyValueMLP) and net.fc1.in_features == 128 and net.fc1.out_features == 256
          and net.fc2.out_features == 256 and net.fc3.out_features == 256 and net.n_actions == 65 and net.raw_width == 72
          and net.fc1.weight.dtype == torch.bfloat16 and net.fc1.weight.is_cuda)
    if not ok:
        raise ValueError("BatchedMatch plays the bf16 128-256-256-256-(65+1) Reversi MLP on a GPU only "
                         "(the net the one-launch search runs)")


class BatchedMatch:
    """``n_games`` (even) games between ``net_a`` and ``net_b``, all searched at once.  ``play()`` returns the result."""

    def __init__(self, net_a, net_b, n_games: int, n_sims: int, n_leaves: int = 4, board_size: int = 8,
                 c_puct: float = 1.25, opening_plies: int = 4, seed: int = 0, first_pair_id: int = 0, device="cuda"):
        n_games, n_sims, n_leaves = int(n_games), int(n_sims), int(n_leaves)
        if n_games <= 0 or n_games % 2 or n_games >= 1 << 16:
            raise ValueError(f"n_games must be even, in 2 .. 65534 (games 2i and 2i+1 are a pair); got {n_games}")
        if n_leaves not in (1, 2, 4):
            raise ValueError(f"n_leaves must be 1, 2 or 4 (the one-launch search); got {n_leaves}")
        if n_sims < n_leaves or n_sims % n_leaves:
            raise ValueError(f"n_sims must be a positive multiple of n_leaves; got {n_sims} and {n_leaves}")
        if board_size not in (4, 6, 8):
            raise ValueError("board_size must be 4, 6 or 8 (Reversi)")
        if opening_plies < 0:
            raise ValueError("opening_plies must be >= 0")
        check_net(net_a)
        check_net(net_b)
        self.net_a, self.net_b = net_a, net_b
        self.n_games, self.n_sims, self.n_leaves, self.board_size = n_games, n_sims, n_leaves, int(board_size)
        self.device = torch.device(device)
        self.n_trees = n_games + TREES_PER_PAIR - 1  # A's range padded to a pair boundary, then B's movers
        self.pools = TreePools(self.n_trees, n_sims, board_size=board_size, c_puct=c_puct, n_leaves=n_leaves,
                               prior_mode=PRIOR_LOGITS_BF16, eval_stride=72, device=device)
        dev, G, T = self.device, n_games, self.n_trees

        def e(n, dt):
            return torch.empty(n, dtype=dt, device=dev)

        self.me, self.opp, self.player, self.ply = e(G, torch.int64), e(G, torch.int64), e(G, torch.int8), e(G, torch.int32)
        self.result, self.count_x, self.count_o = e(G, torch.int8), e(G, torch.uint8), e(G, torch.uint8)
        self.moves, self.tree_of_game = e(G * MAX_PLIES, torch.uint8), e(G, torch.int32)
        self.game_of_tree, self.root_me, self.root_opp = e(T, torch.int32), e(T, torch.int64), e(T, torch.int64)
        self.pair_net = torch.zeros(-(-T // TREES_PER_PAIR), dtype=torch.uint8, device=dev)
        self.counters = torch.zeros(8, dtype=torch.int64, device=dev)
        s = BzMatchState()
        s.n_games, s.board_size, s.opening_plies, s.n_trees = G, self.board_size, int(opening_plies), T
        s.seed, s.first_pair_id = int(seed), int(first_pair_id)
        for name, _ in BzMatchState._fields_[BzMatchState.N_SCALARS:]:
            setattr(s, name, getattr(self, name).data_ptr())
        self.c_struct = s
        self._ref = C.byref(s)
        self._L = _lib.load()
        self.plies = 0
        self.sims = 0
        self.padding = []  # padding trees of every ply
        self._errors = torch.zeros((), dtype=torch.int32, device=dev)  # any tree pool overflow flag of the match

    # -- the steps of a ply -------------------------------------------------------------------------------------------
    def init(self) -> None:
        _lib.check(self._L.bz_match_init(self._ref, _lib.stream_ptr()), "bz_match_init")

    def layout(self) -> tuple[int, int]:
        """the tree layout of this ply; returns (trees to search, padding trees) -- one device-to-host read"""
        _lib.check(self._L.bz_match_layout(self._ref, _lib.stream_ptr()), "bz_match_layout")
        c = self.counters[:3].tolist()
        return int(c[1]), int(c[2])

    def search(self, n_search: int) -> None:
        """reset the first ``n_search`` trees at the layout's roots and search them, each pair with its net"""
        q = BzTreePools.from_buffer_copy(self.pools.c_struct)  # a prefix of the pools: every array starts at tree 0
        q.n_trees = n_search
        ref, st = C.byref(q), _lib.stream_ptr()
        _lib.check(self._L.bz_mcts_reset(ref, _lib.dptr(self.root_me), _lib.dptr(self.root_opp), st), "bz_mcts_reset")
        _lib.check(self._L.bz_mcts_search_fused_two_nets(ref, _lib.dptr(self.net_a._image_pair), _lib.dptr(self.net_b._image_pair),
                                                         _lib.dptr(self.pair_net), self.n_sims // self.n_leaves, st),
                   "bz_mcts_search_fused_two_nets")
        self._errors |= self.pools.error[:n_search].amax()  # stream-ordered: read once, after the match

    def advance(self) -> None:
        _lib.check(self._L.bz_match_advance(self._ref, self.pools._ref, _lib.stream_ptr()), "bz_match_advance")

    # -- the whole match ----------------------------------------------------------------------------------------------
    def play(self) -> dict:
        for n in (self.net_a, self.net_b):
            n.prepare_inference()  # the weight images of the current parameters (in place)
            if getattr(n, "_image_pair", None) is None:
                raise ValueError("the net has no weight image for the one-launch kernel")
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        self.init()
        while True:
            n_search, pad = self.layout()
            if n_search == 0:
                break
            self.search(n_search)
            self.advance()
            self.plies += 1
            self.sims += (n_search - pad) * self.n_sims
            self.padding.append(pad)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        if int(self._errors.item()):
            raise _lib.BzError("tree pool overflow during the match")
        return self.results(wall)

    def results(self, wall_s: float = math.nan) -> dict:
        c = self.counters.tolist()
        result = self.result.cpu()
        a_colour = torch.ones(self.n_games, dtype=torch.int8)
        a_colour[1::2] = -1
        running = result == RUNNING
        for_a = torch.where(running, torch.zeros_like(result), result * a_colour).float()
        pair_scores = ((for_a + 1) / 2).view(-1, 2).mean(1)
        out = {"games": self.n_games, "finished": int(c[3]), "wins": int(c[4]), "draws": int(c[5]), "losses": int(c[6]),
               "disc_diff": int(c[7])}
        out.update(elo_summary(pair_scores[~running.view(-1, 2).any(1)].tolist()))
        out.update({"plies": self.plies, "simulations": self.sims, "wall_s": wall_s,
                    "sims_per_s": self.sims / wall_s if wall_s > 0 else math.nan,
                    "n_sims": self.n_sims, "n_leaves": self.n_leaves, "board_size": self.board_size,
                    "result": result.numpy(), "moves": self.moves.view(self.n_games, MAX_PLIES).cpu().numpy(),
                    "count_x": self.count_x.cpu().numpy(), "count_o": self.count_o.cpu().numpy()})
        return out


def main():
    ap = argparse.ArgumentParser(description="play two checkpoints against each other on one GPU")
    ap.add_argument("--a", required=True, help="checkpoint of net A (train.save_checkpoint)")
    ap.add_argument("--b", required=True, help="checkpoint of net B")
    ap.add_argument("--games", type=int, default=4088, help="even; 4088 games (+ padding) are one launch per ply")
    ap.add_argument("--sims", type=int, default=800)
    ap.add_argument("--leaves", type=int, default=4)
    ap.add_argument("--size", type=int, default=8)
    ap.add_argument("--c-puct", type=float, default=1.25)
    ap.add_argument("--opening-plies", type=int, default=4)
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()
    from . import train

    a, b = train.load_net(args.a), train.load_net(args.b)
    r = BatchedMatch(a, b, args.games, args.sims, n_leaves=args.leaves, board_size=args.size, c_puct=args.c_puct,
                     opening_plies=args.opening_plies, seed=args.seed).play()
    print(json.dumps({k: v for k, v in r.items() if k not in ("result", "moves", "count_x", "count_o")}), flush=True)


if __name__ == "__main__":
    main()
