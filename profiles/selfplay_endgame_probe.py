"""Self-play with the endgame handover on one GPU, at the BASELINE configuration (8x8, 4096 games, 800 simulations, 4
leaves, the bf16 net in the one-launch search, temp_plies 8): feature off, and endgame_empties E in {6, 8, 10, 12} with
a solver phase every K in {1, 8, 32} plies.  --set wld: feature off, the exact handover at E in {10, 12} and the
win/draw/loss handover (endgame_solve="wld") at E in {10, 12, 14}, each with K in {8, 32}.  Per configuration, after --warmup plies (two game lengths: the slots
desynchronise) and over --steps timed plies (about three game lengths, so the waves of finishing games average out):
ms per ply of the search, of the advance and of the solver phases (CUDA events; the phases' share
is spread over the plies), replay records and finished games per second over the --steps timed plies.

    python profiles/selfplay_endgame_probe.py [--set exact|wld] [--out FILE]

The GPU name and power limit are read in the same run and stored with the numbers.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from betazero_b200 import mcts, net, selfplay  # noqa: E402

CONFIGS = {  # (solve, E, K); E = 0: the feature off
    "exact": [("exact", 0, 0)] + [("exact", e, k) for e in (6, 8, 10, 12) for k in (1, 8, 32)],
    "wld": [("exact", 0, 0)] + [("exact", e, k) for e in (10, 12) for k in (8, 32)]
           + [("wld", e, k) for e in (10, 12, 14) for k in (8, 32)],
}


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1],
            "library": os.path.relpath(os.environ.get("BETAZERO_B200_LIB", "betazero_b200/libbetazero_b200.so"),
                                                  os.path.dirname(os.path.dirname(os.path.abspath(__file__))))}


def run(solve: str, empties: int, every: int, args, model) -> dict:
    sp = selfplay.BatchedSelfPlay(args.games, args.sims, mcts.FusedNetEvaluator(model), n_leaves=args.leaves,
                                  temp_plies=8, seed=args.seed, endgame_empties=empties, endgame_every=max(every, 1),
                                  endgame_solve=solve)
    sp.prepare()
    for _ in range(args.warmup):
        sp.play_move()
    sp.drain_replay()  # the timed plies' records fit the buffer (replay_cap = 2 * 128 rows per slot)
    torch.cuda.synchronize()
    s0, eg0 = sp.stats(), (sp.endgame_ms() if empties else 0.0)
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
    for e in ev:
        e[0].record()
        sp.search()
        e[1].record()
        sp.advance()  # with the handover: the solver phase every `every` plies is inside
        e[2].record()
    torch.cuda.synchronize()
    s1, eg1 = sp.stats(), (sp.endgame_ms() if empties else 0.0)
    search = sum(e[0].elapsed_time(e[1]) for e in ev)
    advance_all = sum(e[1].elapsed_time(e[2]) for e in ev)
    phases = eg1 - eg0
    total = ev[0][0].elapsed_time(ev[-1][2])
    recs, games = s1["replay_records"] - s0["replay_records"], s1["games"] - s0["games"]
    assert s1["dropped"] == s0["dropped"], "the replay buffer overflowed: the records per second would be too low"
    n = args.steps
    return {"endgame_solve": solve if empties else None, "endgame_empties": empties or None, "endgame_every": every or None,
            "ms_per_ply": {"search": search / n, "advance": (advance_all - phases) / n, "solver_phases": phases / n,
                           "total": total / n},
            "records_per_s": recs / (total * 1e-3), "games_per_s": games / (total * 1e-3),
            "records": recs, "games_finished": games,
            "endgame_games": s1["endgame_games"] - s0["endgame_games"],
            "endgame_plies": s1["endgame_plies"] - s0["endgame_plies"],
            "endgame_overflow": s1["endgame_overflow"] - s0["endgame_overflow"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=4096)
    ap.add_argument("--sims", type=int, default=800)
    ap.add_argument("--leaves", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=128)
    ap.add_argument("--steps", type=int, default=192)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--set", choices=sorted(CONFIGS), default="exact")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("selfplay_endgame_probe needs a GPU")
    model = net.make_net("mlp", seed=args.seed)
    out = {"gpu": gpu_info(), "config": {k: getattr(args, k) for k in ("games", "sims", "leaves", "warmup", "steps", "set")},
           "runs": []}
    for solve, e, k in CONFIGS[args.set]:
        r = run(solve, e, k, args, model)
        out["runs"].append(r)
        print(json.dumps(r), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f)


if __name__ == "__main__":
    main()
