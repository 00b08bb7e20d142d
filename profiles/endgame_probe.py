"""The endgame solver on one GPU (bz_endgame_solve): 4096 suite positions (betazero_b200.endgame.positions, seed 0) at
8, 10 and 12 empty squares and 512 at 14.  Per set: ms of one call (CUDA events around --repeats calls after a warm-up
call on the first 64 positions), total nodes, nodes per second, the largest and the mean root's nodes.

    python profiles/endgame_probe.py [--out FILE]

The GPU name and power limit are read in the same run and stored with the numbers.  BETAZERO_B200_LIB times another
build of the library (profiles/build_variant.sh): the root split (a -DBZ_SOLVE_SPLIT_PLIES=1 build, since removed)
was timed that way.
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

SETS = [(8, 4096), (10, 4096), (12, 4096), (14, 512)]  # (empties, positions)


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1],
            "library": os.environ.get("BETAZERO_B200_LIB", "betazero_b200/libbetazero_b200.so")}


def time_solve(empties: int, n: int, repeats: int) -> dict:
    s = endgame.positions(n, empties, 8, seed=0)
    minimax.solve(s.me[:64], s.opp[:64], 8)  # warm-up
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(repeats):
        _, _, _, nodes = minimax.solve(s.me, s.opp, 8)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / repeats
    nd = nodes.double()
    return {"empties": empties, "positions": n, "ms_per_call": ms, "nodes": int(nd.sum()),
            "nodes_per_s": float(nd.sum()) / (ms * 1e-3), "max_nodes_per_root": int(nd.max()),
            "mean_nodes_per_root": float(nd.mean())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("endgame_probe needs a GPU")
    out = {"gpu": gpu_info(), "solve": []}
    for empties, n in SETS:
        out["solve"].append(time_solve(empties, n, args.repeats if empties < 14 else 1))
        print(json.dumps(out["solve"][-1]), flush=True)
    print(json.dumps(out), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f)


if __name__ == "__main__":
    main()
