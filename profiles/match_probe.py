"""Net-versus-net match on one GPU: per-ply cost of BatchedMatch against a BatchedSelfPlay ply at the same tree count,
the match driver's own kernels, padding, the whole match, and the sequential arena path for comparison.

    python profiles/match_probe.py [--games 4088] [--sims 800] [--leaves 4] [--out FILE]

Two random-init MLPs (seeds 1 and 2).  Per-ply times are CUDA events; the first 20 plies (every game still live) are
alternated with self-play plies of the same size in the same process.  The GPU name and power limit are read in the
same run and stored with the numbers.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from betazero_b200 import arena, boards, match, mcts, net, players, selfplay  # noqa: E402


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def med(xs):
    return statistics.median(xs) if xs else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=4088)
    ap.add_argument("--sims", type=int, default=800)
    ap.add_argument("--leaves", type=int, default=4)
    ap.add_argument("--arena-games", type=int, default=2)
    ap.add_argument("--out", default=None, help="also write the full result, per-ply rows included, to this JSON file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("match_probe needs a GPU")
    G, S, K = args.games, args.sims, args.leaves
    a, b = net.make_net("mlp", seed=1), net.make_net("mlp", seed=2)
    out = {"gpu": gpu_info(), "games": G, "sims": S, "leaves": K}

    # -- instrumented match, alternated ply by ply with self-play at the same tree count ----------------------------
    m = match.BatchedMatch(a, b, G, S, n_leaves=K, seed=0)
    sp = selfplay.BatchedSelfPlay(G, S, mcts.FusedNetEvaluator(a), n_leaves=K, use_graph=False)
    assert sp.mcts.one_launch
    a.prepare_inference()
    b.prepare_inference()
    for _ in range(2):  # warm-up: lazy initialisation of both paths (sqrt table, shared-memory opt-in)
        sp.play_move()
    m.init()
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    rows = []
    torch.cuda.synchronize()
    t_match = time.perf_counter()
    while True:
        e = [ev() for _ in range(5)]
        t0 = time.perf_counter()
        e[0].record()
        n_search, pad = m.layout()  # ends in the one device-to-host read of the ply: layout_ms holds that round trip
        e[1].record()
        if n_search == 0:
            break
        m.search(n_search)
        e[2].record()
        m.advance()
        e[3].record()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        row = {"ply": m.plies, "trees": n_search, "padding": pad, "live": n_search - pad,
               "ply_ms": e[0].elapsed_time(e[3]), "ply_wall_ms": wall * 1e3,
               "search_ms": e[1].elapsed_time(e[2]), "layout_ms": e[0].elapsed_time(e[1]), "advance_ms": e[2].elapsed_time(e[3])}
        m.plies += 1
        if m.plies <= 20:  # the same process, alternating: a self-play ply of G trees
            e[0].record()
            sp.play_move()
            e[4].record()
            torch.cuda.synchronize()
            row["selfplay_ply_ms"] = e[0].elapsed_time(e[4])
        rows.append(row)
    r = m.results(time.perf_counter() - t_match)
    first = rows[:20]
    out["first_20_plies"] = {
        "match_ply_ms_median": med([x["ply_ms"] for x in first]),
        "match_search_ms_median": med([x["search_ms"] for x in first]),
        "selfplay_ply_ms_median": med([x["selfplay_ply_ms"] for x in first]),
        "layout_plus_advance_ms_median": med([x["layout_ms"] + x["advance_ms"] for x in first]),
        "layout_ms_median": med([x["layout_ms"] for x in first]),
        "advance_ms_median": med([x["advance_ms"] for x in first]),
        "padding_trees": [x["padding"] for x in first],
    }
    out["per_ply"] = rows
    out["padding_trees_mean"] = statistics.mean(x["padding"] for x in rows)

    # -- the whole match, uninstrumented (BatchedMatch.play) ------------------------------------------------------------
    full = match.BatchedMatch(a, b, G, S, n_leaves=K, seed=0).play()
    same = bool((full["moves"] == r["moves"]).all() and (full["result"] == r["result"]).all())
    out["match"] = {k: full[k] for k in ("plies", "simulations", "wall_s", "sims_per_s", "wins", "draws", "losses", "disc_diff",
                                         "score", "elo", "elo_ci", "finished")}
    out["match"]["games_per_s"] = G / full["wall_s"]
    out["match"]["instrumented_run_identical"] = same

    # -- the sequential path: arena.play_match with two MCTSPlayers ---------------------------------------------------
    for p in (a, b):
        p.prepare_inference()
    mk = lambda model: (lambda sym: players.MCTSPlayer(sym, net=model, n_sims=S, n_leaves=K))  # noqa: E731
    arena.play_match(boards.ReversiBoard, mk(a), mk(b), n_games=1)  # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = arena.play_match(boards.ReversiBoard, mk(a), mk(b), n_games=args.arena_games)
    dt = time.perf_counter() - t0
    out["sequential_arena"] = {"games": args.arena_games, "wall_s": dt, "s_per_game": dt / args.arena_games,
                               "games_per_s": args.arena_games / dt, "result": res}
    out["speedup_games_per_s"] = out["match"]["games_per_s"] / out["sequential_arena"]["games_per_s"]
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(out, default=float))
    summary = {k: v for k, v in out.items() if k != "per_ply"}
    print(json.dumps(summary, default=float))


if __name__ == "__main__":
    main()
