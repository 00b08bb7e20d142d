"""Self-play with resignation on one GPU, at the BASELINE configuration (8x8, 4096 games, 800 simulations, 4 leaves, the
bf16 net in the one-launch search, random-init MLP, temp_plies 8).

1. An audit-only run (threshold -1, every game audited): the distribution of q over its records, and the false-positive
   rate FP(v) that each threshold v would have had on its finished games.
2. For thresholds at low quantiles of that distribution, a run with resignation on (resign_audit 0.1), each followed by
   a run with it off: games/s, records/s, plies per finished game, ms per ply of the search and of the advance, and FP
   measured on the run's own audited games.

Per run, after --warmup plies (two game lengths: the slots desynchronise) and over --steps timed plies (CUDA events).

    python profiles/selfplay_resign_probe.py [--out FILE]

The GPU name and power limit are read in the same run and stored with the numbers.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from betazero_b200 import mcts, net, resign, selfplay  # noqa: E402
from profiles.selfplay_endgame_probe import gpu_info  # noqa: E402

QUANTILES = (0.005, 0.01, 0.02, 0.05, 0.1)


def run(threshold, audit: float, args, model) -> tuple[dict, dict]:
    sp = selfplay.BatchedSelfPlay(args.games, args.sims, mcts.FusedNetEvaluator(model), n_leaves=args.leaves,
                                  temp_plies=8, seed=args.seed, resign_threshold=threshold, resign_audit=audit)
    sp.prepare()
    for _ in range(args.warmup):
        sp.play_move()
    sp.drain_replay()  # the timed plies' records fit the buffer (replay_cap = 2 * 128 rows per slot)
    torch.cuda.synchronize()
    s0 = sp.stats()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
    for e in ev:
        e[0].record()
        sp.search()
        e[1].record()
        sp.advance()
        e[2].record()
    torch.cuda.synchronize()
    s1 = sp.stats()
    assert s1["dropped"] == s0["dropped"], "the replay buffer overflowed: the records per second would be too low"
    search = sum(e[0].elapsed_time(e[1]) for e in ev)
    advance = sum(e[1].elapsed_time(e[2]) for e in ev)
    total = ev[0][0].elapsed_time(ev[-1][2])
    recs, games = s1["replay_records"] - s0["replay_records"], s1["games"] - s0["games"]
    n = args.steps
    out = {"threshold": threshold, "audit": audit if threshold is not None else None,
           "ms_per_ply": {"search": search / n, "advance": advance / n, "total": total / n},
           "records_per_s": recs / (total * 1e-3), "games_per_s": games / (total * 1e-3),
           "plies_per_game": recs / games if games else None, "records": recs, "games_finished": games,
           "resigned": s1["resigned"] - s0["resigned"], "audited": s1["audited"] - s0["audited"]}
    records = sp.drain_replay() if threshold is not None else None
    if records is not None:
        records = resign.with_audit(records, args.seed, audit)
        out["audited_games_in_replay"] = resign.audited_games(records)
        out["fp"] = resign.false_positive_rate(records, threshold)
    del sp
    torch.cuda.empty_cache()
    return out, records


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=4096)
    ap.add_argument("--sims", type=int, default=800)
    ap.add_argument("--leaves", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=128)
    ap.add_argument("--steps", type=int, default=192)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("selfplay_resign_probe needs a GPU")
    model = net.make_net("mlp", seed=args.seed)
    out = {"gpu": gpu_info(), "config": {k: getattr(args, k) for k in ("games", "sims", "leaves", "warmup", "steps", "seed")},
           "runs": []}
    off, _ = run(None, 0.1, args, model)
    out["runs"].append(off)
    print(json.dumps(off), flush=True)
    audit_only, recs = run(-1.0, 1.0, args, model)
    q = recs["q"].cpu().numpy()
    q = q[~np.isnan(q)]
    qs = {str(p): float(np.float32(np.quantile(q, p))) for p in QUANTILES + (0.25, 0.5, 0.75, 0.9, 0.99)}
    audit_only["q"] = {"records": int(q.size), "min": float(q.min()), "max": float(q.max()), "mean": float(q.mean()),
                       "quantiles": qs, "histogram": np.histogram(q, bins=20, range=(-1, 1))[0].tolist()}
    audit_only["fp_at_quantiles"] = {str(p): resign.false_positive_rate(recs, qs[str(p)]) for p in QUANTILES}
    audit_only["calibrated"] = {str(t): resign.calibrate(recs, t) for t in (0.01, 0.05, 0.1)}
    out["runs"].append(audit_only)
    print(json.dumps(audit_only), flush=True)
    for p in QUANTILES:
        on, _ = run(qs[str(p)], 0.1, args, model)
        on["quantile"] = p
        out["runs"].append(on)
        print(json.dumps(on), flush=True)
        again, _ = run(None, 0.1, args, model)
        out["runs"].append(again)
        print(json.dumps(again), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f)


if __name__ == "__main__":
    main()
