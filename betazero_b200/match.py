"""Batched net-versus-net matches: thousands of games between two nets on one GPU, every move searched with the
one-launch kernel -- the evaluation the AlphaZero loop needs after an iteration (did the new net get stronger?).

A match is the tournament (``tournament.py``) of two entrants, ``(net_a, n_sims)`` and ``(net_b, n_sims)``, and the one
pairing (0, 1).  Games 2i and 2i+1 form pair i: both start with the same ``opening_plies`` uniformly random legal moves
(Philox keyed by seed, pair id, ply), then net A plays X in game 2i and net B plays X in game 2i+1.  A move is the most
visited root action, lowest action id on ties -- ``MCTSPlayer.get_move`` with the same net, ``n_sims``, ``n_leaves`` and
``c_puct``, so every game can be replayed move for move with the sequential players of ``arena.py``.  Pairs are the
independent unit of the score's interval: the two games of a pair share their opening.

    python -m betazero_b200.match --a A.pt --b B.pt --games 4088 --sims 800 --leaves 4
"""
from __future__ import annotations

import argparse
import json
import math

from .tournament import MAX_PLIES, RUNNING, TREES_PER_PAIR, Minimax, Tournament, check_net, elo, elo_summary  # noqa: F401


class BatchedMatch(Tournament):
    """``n_games`` (even) games between ``net_a`` and ``net_b``, all searched at once.  ``play()`` returns the result.
    ``net_b`` may be ``Minimax(depth)``: net A against the reference's minimax player (a fixed yardstick)."""

    def __init__(self, net_a, net_b, n_games: int, n_sims: int, n_leaves: int = 4, board_size: int = 8,
                 c_puct: float = 1.25, opening_plies: int = 4, seed: int = 0, first_pair_id: int = 0, device="cuda"):
        n_games = int(n_games)
        if n_games <= 0 or n_games % 2 or n_games >= 1 << 16:
            raise ValueError(f"n_games must be even, in 2 .. 65534 (games 2i and 2i+1 are a pair); got {n_games}")
        super().__init__([(net_a, n_sims), net_b if isinstance(net_b, Minimax) else (net_b, n_sims)], n_games, n_leaves=n_leaves, board_size=board_size,
                         c_puct=c_puct, opening_plies=opening_plies, seed=seed, first_pair_id=first_pair_id,
                         device=device)

    def results(self, wall_s: float = math.nan) -> dict:
        r = super().results(wall_s)
        p = r["pairings"][0]
        out = {"games": self.n_games, "finished": r["finished"], "wins": p["wins"], "draws": p["draws"],
               "losses": p["losses"], "disc_diff": int(self.counters[7])}
        out.update({k: p[k] for k in ("score", "elo", "elo_ci", "score_se", "pairs")})
        out.update({k: r[k] for k in ("plies", "simulations", "wall_s", "sims_per_s")})
        out.update({"n_sims": self.n_sims[0], "n_leaves": self.n_leaves, "board_size": self.board_size,
                    "minimax_nodes": r["minimax_nodes"]})
        out.update({k: r[k] for k in ("result", "moves", "count_x", "count_o")})
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
