"""Minimax players on one GPU (one call):

1. bz_minimax_moves on 4096 mid-game 8x8 roots (random playouts of 20..40 plies) at depths 1..6: ms per call (CUDA
   events around --repeats calls after a warm-up), nodes per second, max / mean nodes per root.
2. The ply time of a tournament of a net at 800 simulations (K = 4) against Minimax(4), next to the same net against
   itself: 2 entrants, one pairing, 4088 games; host clock around whole tournaments that end in a device synchronise.

    python profiles/minimax_probe.py [--out FILE]

The GPU name and power limit are read in the same run and stored with the numbers.  BETAZERO_B200_LIB times another
build of the library (profiles/build_variant.sh); the whole-board shape of DESIGN.md section 7 was timed that way.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from betazero_b200 import env, match, minimax, net  # noqa: E402


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1],
            "library": os.environ.get("BETAZERO_B200_LIB", "betazero_b200/libbetazero_b200.so")}


def midgame_roots(n: int, seed: int = 0):
    """mover-relative roots after 20..40 random plies (the game still running)"""
    from oracle import pyoracle as po

    rng = np.random.default_rng(seed)
    me, opp = np.empty(n, np.uint64), np.empty(n, np.uint64)
    i, k = 0, 0
    while i < n:
        g, pl, _, _ = po.random_playout(8, seed * 1_000_003 + k, int(rng.integers(20, 41)))
        k += 1
        m, o = po.grid_to_wire(g, pl)
        if int(po.legal_mask(np.array([m], np.uint64), np.array([o], np.uint64))[0]) == 0:
            continue
        me[i], opp[i] = m, o
        i += 1
    return me, opp


def time_moves(me, opp, depth: int, repeats: int) -> dict:
    keys = torch.arange(me.numel(), dtype=torch.int64, device="cuda")
    a, v, nodes = minimax.best_moves(me, opp, depth, 8, 0, keys)  # warm-up
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(repeats):
        minimax.best_moves(me, opp, depth, 8, 0, keys)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / repeats
    nd = nodes.double()
    return {"depth": depth, "ms_per_call": ms, "nodes": int(nd.sum()), "nodes_per_s": float(nd.sum()) / (ms * 1e-3),
            "max_nodes_per_root": int(nd.max()), "mean_nodes_per_root": float(nd.mean())}


def ply_time(entrant_b, model, games: int, sims: int) -> dict:
    r = None
    for _ in range(2):  # the first run warms up
        r = match.BatchedMatch(model, entrant_b, games, sims, n_leaves=4, seed=1).play()
    return {"plies": r["plies"], "wall_s": r["wall_s"], "ms_per_ply": r["wall_s"] / r["plies"] * 1e3,
            "simulations": r["simulations"], "minimax_nodes": r["minimax_nodes"], "score": r["score"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--roots", type=int, default=4096)
    ap.add_argument("--max-depth", type=int, default=6)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--games", type=int, default=4088)
    ap.add_argument("--sims", type=int, default=800)
    ap.add_argument("--no-tournament", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("minimax_probe needs a GPU")
    out = {"gpu": gpu_info(), "roots": args.roots}
    me_h, opp_h = midgame_roots(args.roots)
    me, opp = env.to_device_u64(me_h), env.to_device_u64(opp_h)
    out["moves"] = []
    for d in range(1, args.max_depth + 1):
        out["moves"].append(time_moves(me, opp, d, args.repeats if d < 6 else max(1, args.repeats // 2)))
        print(json.dumps(out["moves"][-1]), flush=True)
    if not args.no_tournament:
        model = net.make_net("mlp", seed=1)
        out["net_vs_minimax4"] = ply_time(match.Minimax(4), model, args.games, args.sims)
        out["net_vs_itself"] = ply_time(net.make_net("mlp", seed=1), model, args.games, args.sims)
    print(json.dumps(out), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f)


if __name__ == "__main__":
    main()
