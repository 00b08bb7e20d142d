"""The win/draw/loss solve's two levers apart: the ordering threshold T (BZ_SOLVE_ORDER_EMPTIES: fastest-first move
ordering at nodes with at least T empty squares) swept over builds of the library, T = 99 being the null window without
ordering.  Each build is timed by endgame_probe.py --solve wld at 12 (4096 positions) and 14 empties (512), in its own
process (BETAZERO_B200_LIB), and the fastest T (least ms at 12 and 14 together) is reported.

    for t in 6 8 10 12 99; do profiles/build_variant.sh order$t -DBZ_SOLVE_ORDER_EMPTIES=$t; done
    python profiles/endgame_order_sweep.py --thresholds 6,8,10,12,99 [--out FILE] [--best-lib-out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--thresholds", default="6,8,10,12,99")
    ap.add_argument("--lib", default="build/exp/lib_order{t}.so", help="library of threshold {t}")
    ap.add_argument("--out", default=None)
    ap.add_argument("--best-lib-out", default=None, help="write the fastest build's library path here")
    args = ap.parse_args()
    out = {"runs": []}
    for t in (int(x) for x in args.thresholds.split(",")):
        lib = os.path.join(ROOT, args.lib.format(t=t))
        p = subprocess.run([sys.executable, os.path.join(ROOT, "profiles", "endgame_probe.py"), "--solve", "wld",
                            "--empties", "12,14"], env={**os.environ, "BETAZERO_B200_LIB": lib}, capture_output=True,
                           text=True, check=True)
        r = json.loads(p.stdout.strip().splitlines()[-1])
        out["gpu"] = {k: v for k, v in r["gpu"].items() if k != "library"}  # each run names its library
        run = {"order_empties": t, "library": args.lib.format(t=t), "solve": r["solve"],
               "ms_12_plus_14": sum(x["ms_per_call"] for x in r["solve"])}
        out["runs"].append(run)
        print(json.dumps(run), flush=True)
    best = min(out["runs"], key=lambda x: x["ms_12_plus_14"])
    out["best_order_empties"] = best["order_empties"]
    print(json.dumps({"best_order_empties": best["order_empties"], "library": best["library"]}), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f)
    if args.best_lib_out:
        with open(args.best_lib_out, "w") as f:
            f.write(best["library"])


if __name__ == "__main__":
    main()
