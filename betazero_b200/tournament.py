"""Batched round-robin tournaments: every pairing of up to 64 entrants -- a net and a search budget each -- played in the
same launches on one GPU, and one Elo scale fitted over the whole crosstable.  Rates the checkpoints of a training run
(``loop.py --checkpoint 'ckpt/it{iteration}.pt'`` keeps them all) or what search is worth (one net at several budgets).

Pairing k = (i, j) plays ``games_per_pairing`` games, P = games_per_pairing / 2 game pairs: games [2Pk, 2P(k+1)).  Its
game pair p draws its random opening with pair id kP + p, and entrant i is X in the pair's first game and O in its
second -- so pairing k, played alone, is ``BatchedMatch(net_i, net_j, 2P, n_sims, first_pair_id=kP)`` when the two
budgets are equal.  Each ply:

    bz_tournament_layout (each entrant's movers in its own range of whole 56-tree CTA pairs)
    -> bz_mcts_reset -> bz_mcts_search_fused_entrants (each CTA pair loads its entrant's net and runs its budget)
    -> bz_match_advance

A launch lasts as long as its largest budget: the CTA pairs of entrants with smaller budgets finish early and leave
their SMs idle for the rest of it.

An entrant may also be ``Minimax(depth)``: the reference's own opponents, its depth-limited ``OptimalPlayer`` and (depth
0) its ``RandomPlayer`` (reversi_players.py:26-77; ``players.OptimalPlayer``).  They put the nets on a fixed scale: a
checkpoint's rating against ``Minimax(4)`` means the same in every run.  A minimax entrant keeps its range of trees in
the layout but is searched with 0 iterations (its trees are not touched); ``bz_tournament_minimax`` finds its moves
(``bz_minimax_moves`` with the match seed and game key ``2 first_pair_id + g``) and ``bz_tournament_advance`` plays them
next to the nets' most visited actions.  Plies on which no net moves skip the tree search; a tournament of minimax
entrants only allocates no trees at all.

    python -m betazero_b200.tournament A.pt B.pt C.pt --sims 800 --entrant-sims 800,800,200 --games-per-pairing 134
    python -m betazero_b200.tournament A.pt B.pt --minimax 0,2,4
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import time

import numpy as np
import torch

from . import _lib, minimax
from ._lib import BzTournamentState, BzTreePools
from .mcts import PRIOR_LOGITS_BF16, TreePools

TREES_PER_PAIR = 56       # a CTA pair of the one-launch kernel: the unit that loads one net
MAX_PLIES = 128           # BZ_MATCH_MAX_PLIES
RUNNING = 2               # BZ_MATCH_RUNNING
MAX_ENTRANTS = 64         # BZ_MAX_ENTRANTS
LAUNCH_TREES = 148 * 28   # trees of one launch of the one-launch search; more are searched in chunks
Z95 = 1.959963984540054   # two-sided 95 % normal quantile
_C = math.log(10.0) / 400.0


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
        raise ValueError("matches and tournaments play the bf16 128-256-256-256-(65+1) Reversi MLP on a GPU only "
                         "(the net the one-launch search runs)")


def _components(n: int, edges) -> int:
    parent = list(range(n))

    def find(a):
        while parent[a] != a:
            parent[a] = parent[parent[a]]
            a = parent[a]
        return a

    for i, j in edges:
        parent[find(i)] = find(j)
    return len({find(a) for a in range(n)})


def fit_ratings(n_entrants: int, pairings, pair_scores, max_iter: int = 100) -> tuple[np.ndarray, np.ndarray]:
    """Elo ratings of ``n_entrants`` entrants from the game pairs of each pairing; entrant 0 is anchored at 0.

    ``pairings[k] = (i, j)``; ``pair_scores[k]``: the mean score of each of its game pairs from i's view (0 .. 1).
    Model: the logistic Elo model on the pair mean scores, E[s_ij] = 1 / (1 + 10^((r_j - r_i) / 400)), fitted by
    Newton's method on the binomial log-likelihood with the pair as the unit.  Every played pairing gets one virtual
    drawn pair on top of its real ones (n pairs with mean s count as n + 1 pairs with mean (n s + 1/2) / (n + 1)): a
    prior that keeps a clean sweep finite and pulls every rating difference slightly towards 0.  Standard errors come
    from the inverse observed information of that likelihood; a pair's score in [0, 1] with mean p has a variance of at
    most p (1 - p), so they are conservative.  Returns (ratings, standard errors), both [n_entrants].  ValueError if the
    played pairings do not connect every entrant."""
    E = int(n_entrants)
    if E < 1:
        raise ValueError("n_entrants must be >= 1")
    idx_i, idx_j, tot, cnt = [], [], [], []
    for (i, j), xs in zip(pairings, pair_scores):
        xs = np.asarray(xs, dtype=np.float64)
        if not (0 <= i < E and 0 <= j < E) or i == j:
            raise ValueError(f"bad pairing {(i, j)} for {E} entrants")
        if xs.size == 0:
            continue
        idx_i.append(i)
        idx_j.append(j)
        tot.append(float(xs.sum()) + 0.5)  # + the virtual draw
        cnt.append(xs.size + 1.0)
    if _components(E, zip(idx_i, idx_j)) != 1:
        raise ValueError("the played pairings do not connect all entrants: their ratings are not on one scale")
    ii, jj, S, N = np.array(idx_i, int), np.array(idx_j, int), np.array(tot), np.array(cnt)
    r = np.zeros(E)

    def loglik(r):
        d = (r[ii] - r[jj]) * _C
        return float(np.sum(S * -np.logaddexp(0.0, -d) + (N - S) * -np.logaddexp(0.0, d)))

    def info(r):
        p = 1.0 / (1.0 + np.exp(-(r[ii] - r[jj]) * _C))
        g = np.zeros(E)
        np.add.at(g, ii, (S - N * p) * _C)
        np.add.at(g, jj, -(S - N * p) * _C)
        w = N * p * (1.0 - p) * _C * _C
        H = np.zeros((E, E))
        np.add.at(H, (ii, ii), w)
        np.add.at(H, (jj, jj), w)
        np.add.at(H, (ii, jj), -w)
        np.add.at(H, (jj, ii), -w)
        return g, H

    if E > 1:
        ll = loglik(r)
        for _ in range(max_iter):
            g, H = info(r)
            step = np.zeros(E)
            step[1:] = np.linalg.solve(H[1:, 1:], g[1:])
            t = 1.0
            while True:  # Newton step, halved while it lowers the (concave) likelihood
                nr = r + t * step
                nll = loglik(nr)
                if nll >= ll or t < 1e-6:
                    break
                t *= 0.5
            r, ll = nr, nll
            if np.max(np.abs(t * step)) < 1e-10:
                break
    se = np.zeros(E)
    if E > 1:
        _, H = info(r)
        se[1:] = np.sqrt(np.diag(np.linalg.inv(H[1:, 1:])))
    return r, se


class Minimax:
    """A tournament entrant that plays the reference's depth-limited minimax ``OptimalPlayer`` (``depth`` 0 .. 8; 0 is
    its ``RandomPlayer``): in a ``Tournament``'s entrant list in place of ``(net, n_sims)``, or as ``BatchedMatch``'s B."""

    def __init__(self, depth: int):
        self.depth = minimax.check_depth(depth)

    def __repr__(self):
        return f"Minimax({self.depth})"


class Tournament:
    """Every pairing of ``entrants`` -- a list of ``(net, n_sims)`` and ``Minimax(depth)``; one net may appear with
    several budgets and then shares its weight image -- for ``games_per_pairing`` (even) games, all searched at once.
    ``play()`` returns the result.  Game pair i draws its opening with pair id ``first_pair_id + i``."""

    def __init__(self, entrants, games_per_pairing: int, n_leaves: int = 4, board_size: int = 8, c_puct: float = 1.25,
                 opening_plies: int = 4, seed: int = 0, pairings=None, first_pair_id: int = 0, device="cuda"):
        entrants = list(entrants)
        E = len(entrants)
        if not 2 <= E <= MAX_ENTRANTS:
            raise ValueError(f"a tournament has 2 .. {MAX_ENTRANTS} entrants; got {E}")
        n_leaves, gpp = int(n_leaves), int(games_per_pairing)
        if n_leaves not in (1, 2, 4):
            raise ValueError(f"n_leaves must be 1, 2 or 4 (the one-launch search); got {n_leaves}")
        depths = [x.depth if isinstance(x, Minimax) else -1 for x in entrants]  # -1: a net entrant
        sims = [0 if d >= 0 else int(x[1]) for x, d in zip(entrants, depths)]
        for s, d in zip(sims, depths):
            if d < 0 and (s < n_leaves or s % n_leaves):
                raise ValueError(f"every budget must be a positive multiple of n_leaves; got {s} and {n_leaves}")
        if gpp <= 0 or gpp % 2:
            raise ValueError(f"games_per_pairing must be even and positive (games are played in pairs); got {gpp}")
        if board_size not in (4, 6, 8):
            raise ValueError("board_size must be 4, 6 or 8 (Reversi)")
        if opening_plies < 0:
            raise ValueError("opening_plies must be >= 0")
        if pairings is None:
            pairings = [(i, j) for i in range(E) for j in range(i + 1, E)]
        pairings = [(int(i), int(j)) for i, j in pairings]
        seen = set()
        for i, j in pairings:
            if not (0 <= i < E and 0 <= j < E) or i == j:
                raise ValueError(f"pairing {(i, j)}: two different entrants of 0 .. {E - 1}")
            if frozenset((i, j)) in seen:
                raise ValueError(f"pairing {(i, j)} appears twice")
            seen.add(frozenset((i, j)))
        if _components(E, pairings) != 1:
            raise ValueError("the pairings do not connect all entrants: their ratings would not be on one scale")
        n_games = len(pairings) * gpp
        if n_games >= 1 << 16:
            raise ValueError(f"{n_games} games in all; a tournament holds fewer than 65536")
        nets = []  # distinct nets, in order of first appearance
        for x, d in zip(entrants, depths):
            n = x[0] if d < 0 else None
            if n is not None and not any(n is m for m in nets):
                check_net(n)
                nets.append(n)
        self.entrants, self.nets, self.pairings = entrants, nets, pairings
        self.n_entrants, self.n_sims, self.n_leaves, self.board_size = E, sims, n_leaves, int(board_size)
        self.depths = depths
        self.games_per_pairing, self.n_games = gpp, n_games
        self.device = torch.device(device)
        self.n_trees = n_games + (TREES_PER_PAIR - 1) * (E - 1)  # every range but the last padded to a pair boundary
        self.pools = (TreePools(self.n_trees, max(sims), board_size=board_size, c_puct=c_puct, n_leaves=n_leaves,
                                prior_mode=PRIOR_LOGITS_BF16, eval_stride=72, device=device) if nets else None)
        dev, G, T = self.device, n_games, self.n_trees

        def e(n, dt):
            return torch.empty(n, dtype=dt, device=dev)

        self.me, self.opp, self.player, self.ply = e(G, torch.int64), e(G, torch.int64), e(G, torch.int8), e(G, torch.int32)
        self.result, self.count_x, self.count_o = e(G, torch.int8), e(G, torch.uint8), e(G, torch.uint8)
        self.moves, self.tree_of_game = e(G * MAX_PLIES, torch.uint8), e(G, torch.int32)
        self.game_of_tree, self.root_me, self.root_opp = e(T, torch.int32), e(T, torch.int64), e(T, torch.int64)
        self.pair_net = torch.zeros(-(-T // TREES_PER_PAIR), dtype=torch.uint8, device=dev)  # entrant of each CTA pair
        self.counters = torch.zeros(8, dtype=torch.int64, device=dev)
        P = gpp // 2
        self.pairing_of_pair = np.repeat(np.arange(len(pairings)), P)
        pi = np.array(pairings, dtype=np.uint8).reshape(-1, 2)
        self.first = torch.from_numpy(pi[self.pairing_of_pair, 0].copy()).to(dev)
        self.second = torch.from_numpy(pi[self.pairing_of_pair, 1].copy()).to(dev)
        s = BzTournamentState()
        m = s.match
        m.n_games, m.board_size, m.opening_plies, m.n_trees = G, self.board_size, int(opening_plies), T
        m.seed, m.first_pair_id = int(seed), int(first_pair_id)
        for name, _ in m._fields_[m.N_SCALARS:]:
            setattr(m, name, getattr(self, name).data_ptr())
        s.n_entrants, s.first, s.second = E, self.first.data_ptr(), self.second.data_ptr()
        self.opening_plies = int(opening_plies)
        self.c_struct = s
        self._ref, self._mref = C.byref(s), C.byref(s.match)
        self._images = (C.c_void_p * E)()
        self._iters = (C.c_int32 * E)(*[x // n_leaves for x in sims])
        self._depths = (C.c_int32 * E)(*depths)
        self.has_minimax = any(d >= 0 for d in depths)
        if self.has_minimax:
            self.minimax_action = e(T, torch.uint8)
            self.minimax_nodes = torch.zeros(1, dtype=torch.int64, device=dev)
            self._minimax_ws = minimax.workspace(T, dev)
        self._net_moves = self._minimax_moves = bool(nets)  # who moves this ply (layout)
        self._L = _lib.load()
        self.plies = 0
        self.padding, self.chunks = [], []  # padding trees and launches of every ply
        self._errors = torch.zeros((), dtype=torch.int32, device=dev)  # any tree pool overflow flag of the tournament

    # -- the steps of a ply -------------------------------------------------------------------------------------------
    def init(self) -> None:
        """the openings; the entrants' weight images (``prepare_inference``) must exist"""
        for k, (x, d) in enumerate(zip(self.entrants, self.depths)):
            # a minimax entrant runs 0 iterations and loads no weights, but the entry wants an image for it
            self._images[k] = (x[0] if d < 0 else self.nets[0])._image_pair.data_ptr() if self.nets else None
        if self.has_minimax:
            self.minimax_nodes.zero_()
        _lib.check(self._L.bz_match_init(self._mref, _lib.stream_ptr()), "bz_match_init")

    def layout(self) -> tuple[int, int]:
        """the tree layout of this ply; returns (trees to search, padding trees) -- one device-to-host read"""
        _lib.check(self._L.bz_tournament_layout(self._ref, _lib.stream_ptr()), "bz_tournament_layout")
        if not self.has_minimax:
            c = self.counters[:3].tolist()
            return int(c[1]), int(c[2])
        if not self.nets:
            c = self.counters[:3].tolist()
            self._net_moves, self._minimax_moves = False, c[1] > 0
            return int(c[1]), int(c[2])
        c = torch.cat((self.counters[:3], self.pair_net.to(torch.int64))).tolist()
        movers = {self.depths[e] >= 0 for e in c[3:3 + -(-int(c[1]) // TREES_PER_PAIR)]}
        self._net_moves, self._minimax_moves = False in movers, True in movers
        return int(c[1]), int(c[2])

    def search(self, n_search: int) -> None:
        """reset the first ``n_search`` trees at the layout's roots and search them, each CTA pair as its entrant (nothing
        on a ply where no net moves)"""
        if not self._net_moves:
            return
        q = BzTreePools.from_buffer_copy(self.pools.c_struct)  # a prefix of the pools: every array starts at tree 0
        q.n_trees = n_search
        ref, st = C.byref(q), _lib.stream_ptr()
        _lib.check(self._L.bz_mcts_reset(ref, _lib.dptr(self.root_me), _lib.dptr(self.root_opp), st), "bz_mcts_reset")
        _lib.check(self._L.bz_mcts_search_fused_entrants(ref, self._images, self._iters, self.n_entrants,
                                                         _lib.dptr(self.pair_net), st), "bz_mcts_search_fused_entrants")
        self._errors |= self.pools.error[:n_search].amax()  # stream-ordered: read once, after the tournament

    def minimax_search(self) -> None:
        """the minimax entrants' moves of this ply"""
        if self.has_minimax and self._minimax_moves:
            _lib.check(self._L.bz_tournament_minimax(self._ref, self._depths, _lib.dptr(self._minimax_ws),
                                                     _lib.dptr(self.minimax_action), _lib.dptr(self.minimax_nodes),
                                                     _lib.stream_ptr()), "bz_tournament_minimax")

    def advance(self) -> None:
        if not self.has_minimax:
            _lib.check(self._L.bz_match_advance(self._mref, self.pools._ref, _lib.stream_ptr()), "bz_match_advance")
            return
        _lib.check(self._L.bz_tournament_advance(self._ref, self.pools._ref if self.pools else None, self._depths,
                                                 _lib.dptr(self.minimax_action), _lib.stream_ptr()),
                   "bz_tournament_advance")

    # -- the whole tournament -----------------------------------------------------------------------------------------
    def play(self) -> dict:
        for n in self.nets:
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
            self.minimax_search()
            self.advance()
            self.plies += 1
            self.padding.append(pad)
            self.chunks.append(-(-n_search // LAUNCH_TREES))
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        if self.pools is not None and int(self._errors.item()):
            raise _lib.BzError("tree pool overflow during the tournament")
        return self.results(wall)

    def results(self, wall_s: float = math.nan) -> dict:
        G, E = self.n_games, self.n_entrants
        result = self.result.cpu().numpy().astype(np.int64)
        moves = self.moves.view(G, MAX_PLIES).cpu().numpy()
        pairing = np.repeat(self.pairing_of_pair, 2)
        first, second = self.first.cpu().numpy()[np.arange(G) // 2], self.second.cpu().numpy()[np.arange(G) // 2]
        x_ent = np.where(np.arange(G) % 2 == 0, first, second)
        o_ent = np.where(np.arange(G) % 2 == 0, second, first)
        # simulations: every recorded move after the opening was searched by the entrant to move, with its budget (0 for a
        # minimax entrant)
        budget = np.array(self.n_sims)
        k = np.arange(MAX_PLIES)[None, :]
        searched = (moves != 255) & (k >= self.opening_plies)
        mover = np.where(k % 2 == 0, x_ent[:, None], o_ent[:, None])
        sims = int((budget[mover] * searched).sum())
        running = result == RUNNING
        for_first = np.where(running, 0, result * np.where(np.arange(G) % 2 == 0, 1, -1))
        score = (for_first + 1) / 2.0
        pair_score, pair_done = score.reshape(-1, 2).mean(1), ~running.reshape(-1, 2).any(1)
        cross = np.full((E, E), math.nan)
        per, scores = [], []
        for kk, (i, j) in enumerate(self.pairings):
            g = pairing == kk
            done = g & ~running
            ps = pair_score[(self.pairing_of_pair == kk) & pair_done]
            scores.append(ps)
            d = {"i": i, "j": j, "n_sims_i": self.n_sims[i], "n_sims_j": self.n_sims[j],
                 "wins": int((for_first[done] > 0).sum()), "draws": int((for_first[done] == 0).sum()),
                 "losses": int((for_first[done] < 0).sum())}
            d.update(elo_summary(ps.tolist()))
            per.append(d)
            if done.any():
                cross[i, j] = float(score[done].mean())
                cross[j, i] = 1.0 - cross[i, j]
        ratings, se = fit_ratings(E, self.pairings, scores)
        pads = np.array(self.padding, dtype=np.float64)
        return {"entrants": E, "n_sims": list(self.n_sims), "n_leaves": self.n_leaves, "board_size": self.board_size,
                "games": G, "games_per_pairing": self.games_per_pairing, "finished": int((~running).sum()),
                "pairings": per, "crosstable": cross.tolist(), "ratings": ratings.tolist(), "rating_se": se.tolist(),
                "plies": self.plies, "simulations": sims, "wall_s": wall_s,
                "kinds": ["minimax" if d >= 0 else "net" for d in self.depths],
                "depths": [d if d >= 0 else None for d in self.depths],
                "minimax_nodes": int(self.minimax_nodes.item()) if self.has_minimax else 0,
                "sims_per_s": sims / wall_s if wall_s > 0 else math.nan,
                "padding_per_ply": float(pads.mean()) if pads.size else 0.0,
                "max_padding": int(pads.max()) if pads.size else 0,
                "chunks_per_ply": max(self.chunks, default=0),
                "pairing": pairing, "result": result.astype(np.int8), "moves": moves,
                "count_x": self.count_x.cpu().numpy(), "count_o": self.count_o.cpu().numpy()}


PER_GAME = ("pairing", "result", "moves", "count_x", "count_o")


def main():
    ap = argparse.ArgumentParser(description="a round-robin tournament between checkpoints on one GPU")
    ap.add_argument("checkpoints", nargs="*", help="checkpoints (train.save_checkpoint); one entrant each, a path may repeat")
    ap.add_argument("--minimax", default=None, help="comma-separated depths (0 .. 8): one minimax entrant each, after the "
                                                    "checkpoints (the reference's OptimalPlayer; depth 0 is its RandomPlayer)")
    ap.add_argument("--sims", type=int, default=800, help="simulations per move of every entrant")
    ap.add_argument("--entrant-sims", default=None, help="comma-separated simulations per move, one per entrant (overrides --sims)")
    ap.add_argument("--games-per-pairing", type=int, default=134, help="even; 28 pairings x 134 games fit one launch per ply")
    ap.add_argument("--leaves", type=int, default=4)
    ap.add_argument("--size", type=int, default=8)
    ap.add_argument("--c-puct", type=float, default=1.25)
    ap.add_argument("--opening-plies", type=int, default=4)
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()
    sims = [int(x) for x in args.entrant_sims.split(",")] if args.entrant_sims else [args.sims] * len(args.checkpoints)
    if len(sims) != len(args.checkpoints):
        raise SystemExit(f"--entrant-sims lists {len(sims)} budgets for {len(args.checkpoints)} entrants")
    from . import train

    loaded = {}
    for p in args.checkpoints:
        if p not in loaded:
            loaded[p] = train.load_net(p)
    entrants = [(loaded[p], s) for p, s in zip(args.checkpoints, sims)]
    entrants += [Minimax(int(d)) for d in args.minimax.split(",")] if args.minimax else []
    r = Tournament(entrants, args.games_per_pairing, n_leaves=args.leaves,
                   board_size=args.size, c_puct=args.c_puct, opening_plies=args.opening_plies, seed=args.seed).play()
    r["checkpoints"] = args.checkpoints
    r["minimax"] = [e.depth for e in entrants if isinstance(e, Minimax)]
    print(json.dumps({k: v for k, v in r.items() if k not in PER_GAME}), flush=True)


if __name__ == "__main__":
    main()
