"""The endgame solver on one GPU (bz_endgame_solve, and with --solve wld or both bz_endgame_solve_wld): 4096 suite
positions (betazero_b200.endgame.positions, seed 0) at 8, 10 and 12 empty squares and 512 at 14.  Per set and solve: ms
of one call (CUDA events around --repeats calls after a warm-up call on the first 64 positions; one call from 14
empties on), total nodes, nodes per second, the largest and the mean root's nodes.

    python profiles/endgame_probe.py [--solve exact|wld|both] [--empties 8,10,12,14,16,18,20] [--out FILE]

Past 14 empties (the win/draw/loss solve only) nobody knew the cost, so a set starts with 16 positions and is scaled up
from the measured time, towards --budget-s seconds a call (at most 4096 positions); every count run is reported.  A set
is skipped, and reported as such, when the growth from the set two empties below predicts more than --budget-s seconds
for 16 positions.

The GPU name and power limit are read in the same run and stored with the numbers.  BETAZERO_B200_LIB times another
build of the library (profiles/build_variant.sh): the root split (a -DBZ_SOLVE_SPLIT_PLIES=1 build, since removed) and
the win/draw/loss solve's ordering threshold (-DBZ_SOLVE_ORDER_EMPTIES=T, endgame_order_sweep.py) were timed that way.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from betazero_b200 import endgame, minimax  # noqa: E402

SETS = {8: 4096, 10: 4096, 12: 4096, 14: 512}  # empties -> positions; past 14: scaled from 16


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1],
            "library": os.path.relpath(os.environ.get("BETAZERO_B200_LIB", "betazero_b200/libbetazero_b200.so"),
                                                  os.path.dirname(os.path.dirname(os.path.abspath(__file__))))}


def time_solve(empties: int, n: int, repeats: int, wld: bool = False, suite=None, warm: bool = True) -> dict:
    s = suite if suite is not None else endgame.positions(n, empties, 8, seed=0)
    me, opp = s.me[:n], s.opp[:n]
    if warm:  # the scaled sets skip it: their first 64 positions can take as long as the call
        minimax.solve(me[:64], opp[:64], 8, wld=wld)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(repeats):
        _, _, _, nodes = minimax.solve(me, opp, 8, wld=wld)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / repeats
    nd = nodes.double()
    return {"solve": "wld" if wld else "exact", "empties": empties, "positions": n, "ms_per_call": ms,
            "nodes": int(nd.sum()), "nodes_per_s": float(nd.sum()) / (ms * 1e-3), "max_nodes_per_root": int(nd.max()),
            "mean_nodes_per_root": float(nd.mean())}


def scaled_runs(empties: int, budget_s: float, base: dict) -> list:
    """the win/draw/loss solve past 14 empties: 16 positions, then more while a call stays under a quarter of the budget
    (the count scaled by the measured time, at most 16x a step and 4096 in all).  base: the 16-position call two empties
    below; with its own growth it predicts this set's first call, and a prediction above the budget skips the set."""
    if base.get("growth"):
        predicted = base["ms_per_call"] * base["growth"] * 1e-3
        if predicted > budget_s:
            return [{"solve": "wld", "empties": empties, "positions": 16, "ms_per_call": None,
                     "skipped": f"predicted {predicted:.0f} s for 16 positions (x{base['growth']:.1f} per two empties), "
                                f"above the {budget_s:.0f} s budget"}]
    s = endgame.positions(16, empties, 8, seed=0)
    runs, n = [], 16
    while True:
        if s.me.numel() < n:
            s = endgame.positions(n, empties, 8, seed=0)  # the same seed: the first positions are the same
        r = time_solve(empties, n, 1, wld=True, suite=s, warm=False)
        if n == 16:
            r["growth"] = r["ms_per_call"] / base["ms_per_call"]  # per two empties, 16 positions
        runs.append(r)
        print(json.dumps(r), flush=True)
        t = r["ms_per_call"] * 1e-3
        if t > budget_s / 4 or n >= 4096:
            return runs
        n = min(4096, n * max(2, min(16, int(budget_s / 4 / max(t, 1e-3)))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--solve", choices=("exact", "wld", "both"), default="exact")
    ap.add_argument("--empties", default="8,10,12,14", help="sets, comma-separated; past 14 the wld solve only")
    ap.add_argument("--budget-s", type=float, default=40.0, help="past 14 empties: the longest call to aim for")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("endgame_probe needs a GPU")
    modes = {"exact": [False], "wld": [True], "both": [False, True]}[args.solve]
    out = {"gpu": gpu_info(), "solve": []}
    base = None  # the wld solve's 16-position call two empties below (scaled sets)
    for empties in sorted(int(x) for x in args.empties.split(",")):
        if empties in SETS:
            for wld in modes:
                out["solve"].append(time_solve(empties, SETS[empties], args.repeats if empties < 14 else 1, wld))
                print(json.dumps(out["solve"][-1]), flush=True)
            continue
        if True not in modes:
            raise SystemExit(f"{empties} empties: only the wld solve is timed past 14")
        if base is None or base["empties"] != empties - 2:
            base = time_solve(empties - 2, 16, 1, wld=True, warm=False)
            base["role"] = "growth base"
            out["solve"].append(base)
            print(json.dumps(base), flush=True)
        if base["ms_per_call"] is None:  # the set below was skipped: so is this one
            out["solve"].append({"solve": "wld", "empties": empties, "positions": 16, "ms_per_call": None,
                                 "skipped": f"the set at {empties - 2} empties was skipped"})
            base = dict(out["solve"][-1])
            continue
        runs = scaled_runs(empties, args.budget_s, base)
        out["solve"] += runs
        base = runs[0]
    print(json.dumps(out), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f)


if __name__ == "__main__":
    main()
