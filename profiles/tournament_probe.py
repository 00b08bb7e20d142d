"""Round-robin tournament on one GPU: 8 entrants -- four random-init MLPs (seeds 1..4), each at 800 and at 200
simulations per move -- all 28 pairings x 134 games (3752 games, K = 4 leaves per iteration).  With at most 7 x 55
padding trees every ply fits one launch (3752 + 385 <= 4144 trees).

    python profiles/tournament_probe.py [--out FILE]

Compared in the same process: a BatchedMatch of 3752 games at 800 simulations (the same tree count: a tournament of two
entrants, one net pair), and the same tournament with every budget at 800, which isolates what mixed budgets cost: a
launch lasts as long as its largest budget, so the pairs of 200-simulation entrants idle for the rest of it.  Every
configuration runs once as a warm-up, then --repeats times; wall times are host clocks around work that ends in a device
synchronise.  The GPU name and power limit are read in the same run and stored with the numbers.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from betazero_b200 import match, net, tournament  # noqa: E402


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def summary(r: dict) -> dict:
    out = {k: r[k] for k in ("plies", "simulations", "wall_s", "sims_per_s") if k in r}
    out["ms_per_ply"] = r["wall_s"] / r["plies"] * 1e3 if r["plies"] else None
    for k in ("padding_per_ply", "max_padding", "chunks_per_ply", "ratings", "rating_se"):
        if k in r:
            out[k] = r[k]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games-per-pairing", type=int, default=134)
    ap.add_argument("--sims", type=int, default=800)
    ap.add_argument("--low-sims", type=int, default=200)
    ap.add_argument("--leaves", type=int, default=4)
    ap.add_argument("--repeats", type=int, default=2)
    ap.add_argument("--out", default=None, help="also write the result to this JSON file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("tournament_probe needs a GPU")
    S, L, K = args.sims, args.low_sims, args.leaves
    nets = [net.make_net("mlp", seed=s) for s in (1, 2, 3, 4)]
    mixed = [(n, s) for n in nets for s in (S, L)]  # entrant 2k: net k at S, entrant 2k + 1: net k at L
    equal = [(n, S) for n in nets for _ in range(2)]
    gpp = args.games_per_pairing
    G = 28 * gpp
    out = {"gpu": gpu_info(), "entrants": 8, "pairings": 28, "games_per_pairing": gpp, "games": G, "leaves": K,
           "budgets_mixed": [s for _, s in mixed], "budgets_equal": [s for _, s in equal]}
    runs = {
        "tournament_mixed": lambda: tournament.Tournament(mixed, gpp, n_leaves=K).play(),
        "tournament_equal": lambda: tournament.Tournament(equal, gpp, n_leaves=K).play(),
        "match": lambda: match.BatchedMatch(nets[0], nets[1], G, S, n_leaves=K).play(),
    }
    for name, fn in runs.items():
        fn()  # warm-up
    for name, fn in runs.items():
        rs = [fn() for _ in range(args.repeats)]
        out[name] = summary(min(rs, key=lambda r: r["wall_s"]))
        out[name]["wall_s_all"] = [r["wall_s"] for r in rs]
    t, e, m = out["tournament_mixed"], out["tournament_equal"], out["match"]
    out["mixed_vs_equal_ms_per_ply"] = t["ms_per_ply"] / e["ms_per_ply"]
    out["mixed_vs_equal_sims_per_s"] = t["sims_per_s"] / e["sims_per_s"]
    out["equal_vs_match_sims_per_s"] = e["sims_per_s"] / m["sims_per_s"]
    out["rating_800_minus_200_mean"] = statistics.mean(t["ratings"][2 * k] - t["ratings"][2 * k + 1] for k in range(4))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(out, default=float))
    print(json.dumps(out, default=float))


if __name__ == "__main__":
    main()
