"""Self-play with randomized search budgets on one GPU: 8x8, 4 leaves, 800 simulations, the bf16 net (random-init MLP) in
the one-launch search, temp_plies 8, at 4096 and 16 384 games.

Configurations: off (every ply at 800), p = 0.25 with fast_sims 160, p = 0.2 with fast_sims 160.  The three drivers of a
size live in one process and take turns: each turn runs warm-up plies (--first-warmup on a driver's first turn,
--warmup after), then --steps timed plies (CUDA events around
every ply and the whole window), and the sizes' turns repeat --repeats times.  Per turn: ms per ply, games finished per
second, full records per second (records with full = 1 flushed during the window), library launches per ply, and for the
randomized runs the share of plies whose full range (full trees padded to a CTA pair) ends past the first launch's trees
(the one-launch search holds 4144 trees; more are searched in equal chunks of whole CTA pairs).  The layout kernel is
timed on its own afterwards (--layout-reps launches between two events).

    python profiles/selfplay_cap_probe.py [--out FILE]

The GPU name and power limit are read in the same run and stored with the numbers.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from betazero_b200 import _lib, mcts, net, selfplay  # noqa: E402
from profiles.selfplay_endgame_probe import gpu_info  # noqa: E402

CONFIGS = [("off", None, None), ("p0.25_f160", 0.25, 160), ("p0.2_f160", 0.2, 160)]
MAX_TREES = mcts.BatchedMCTS.ONE_LAUNCH_MAX_TREES


def first_chunk_trees(n_trees: int) -> int:
    """the trees of the first launch of bz_mcts_search_fused(_entrants): equal chunks of whole CTA pairs"""
    n_chunks = -(-n_trees // MAX_TREES)
    return -(-(-(-n_trees // n_chunks)) // 112) * 112


def turn(sp, args, warmup: int) -> dict:
    for _ in range(warmup):
        sp.play_move()
    sp.drain_replay()
    torch.cuda.synchronize()
    s0, l0 = sp.stats(), sp.total_launches()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(args.steps)]
    full_trees = []
    for e in ev:
        e[0].record()
        sp.play_move()
        e[1].record()
        if sp.cs is not None:  # the full range's end of this ply (a tiny reduction, no host synchronisation)
            full_trees.append((sp.pair_entrant == 0).sum())
    torch.cuda.synchronize()
    s1, l1 = sp.stats(), sp.total_launches()
    assert s1["dropped"] == s0["dropped"], "the replay buffer overflowed"
    total = ev[0][0].elapsed_time(ev[-1][1])
    plies = [e[0].elapsed_time(e[1]) for e in ev]
    rp = sp.drain_replay()
    n_rec = int(rp["me"].shape[0])
    full_rec = int(rp["full"].sum()) if "full" in rp else n_rec
    games = s1["games"] - s0["games"]
    out = {"ms_per_ply": total / args.steps, "ms_per_ply_min": min(plies), "ms_per_ply_max": max(plies),
           "games_per_s": games / (total * 1e-3), "full_records_per_s": full_rec / (total * 1e-3),
           "records_per_s": n_rec / (total * 1e-3), "games_finished": games, "records": n_rec, "full_records": full_rec,
           "launches_per_ply": (l1 - l0) / args.steps}
    if sp.cs is not None:
        ft = torch.stack(full_trees).cpu() * 56
        limit = first_chunk_trees(sp.pools.n_trees)
        out.update({"full_plies": s1["full_plies"] - s0["full_plies"], "fast_plies": s1["fast_plies"] - s0["fast_plies"],
                    "full_trees_mean": float(ft.double().mean()), "full_trees_max": int(ft.max()),
                    "first_launch_trees": limit, "plies_full_range_past_first_launch": int((ft > limit).sum())})
    return out


def layout_ms(sp, reps: int) -> float:
    st = _lib.stream_ptr()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(16):
        _lib.check(sp._L.bz_selfplay_cap_layout(sp._ref, sp._cs_ref, st), "bz_selfplay_cap_layout")
    t0.record()
    for _ in range(reps):
        _lib.check(sp._L.bz_selfplay_cap_layout(sp._ref, sp._cs_ref, st), "bz_selfplay_cap_layout")
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, nargs="+", default=[4096, 16384])
    ap.add_argument("--sims", type=int, default=800)
    ap.add_argument("--leaves", type=int, default=4)
    ap.add_argument("--first-warmup", type=int, default=128, help="plies before a driver's first window (two game "
                                                                   "lengths: the slots desynchronise)")
    ap.add_argument("--warmup", type=int, default=16, help="plies before every later window")
    ap.add_argument("--steps", type=int, default=64)
    ap.add_argument("--repeats", type=int, default=2)
    ap.add_argument("--layout-reps", type=int, default=200)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("selfplay_cap_probe needs a GPU")
    model = net.make_net("mlp", seed=args.seed)
    out = {"gpu": gpu_info(), "config": {k: getattr(args, k) for k in ("games", "sims", "leaves", "first_warmup", "warmup",
                                                                       "steps", "repeats", "seed")}, "runs": []}
    for B in args.games:
        sps = {name: selfplay.BatchedSelfPlay(B, args.sims, mcts.FusedNetEvaluator(model), n_leaves=args.leaves,
                                              temp_plies=8, seed=args.seed, fast_sims=fast,
                                              full_fraction=p if p is not None else 0.25)
               for name, p, fast in CONFIGS}
        for sp in sps.values():
            sp.prepare()
        for rep in range(args.repeats):
            for name, p, fast in CONFIGS:
                r = {"games": B, "config": name, "full_fraction": p, "fast_sims": fast, "repeat": rep,
                     **turn(sps[name], args, args.first_warmup if rep == 0 else args.warmup)}
                out["runs"].append(r)
                print(json.dumps(r), flush=True)
        for name, p, _ in CONFIGS:
            if p is not None:
                r = {"games": B, "config": name, "layout_kernel_ms": layout_ms(sps[name], args.layout_reps)}
                out["runs"].append(r)
                print(json.dumps(r), flush=True)
        del sps
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f)


if __name__ == "__main__":
    main()
