#!/usr/bin/env python
"""bench.py -- Reversi 8x8 self-play MCTS throughput on B200 (BASELINE.json's headline metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA engine
    python bench.py --impl reference --steps K --warmup W     # the CPU arm (oracle port) on host cores
    torchrun --nproc-per-node N ... bench.py --gpus N ...     # one rank per GPU (games shard, no collective)
    python bench.py ... --dump-outputs DIR                    # also write the last timed step's outputs (rank 0)

A "step" is one lockstep ply of self-play for every game of the rank: one batched MCTS of
``--sims`` iterations over ``--games`` concurrent trees (select -> gather -> net -> expand/backup,
every iteration) followed by the move/terminal/replay kernel.  Workload at N=1: BASELINE config
"Reversi 8x8 self-play, 800 sims/move, 4096 games per GPU".  One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "reversi8x8_selfplay_mcts_sims_per_sec"
UNIT = "sims/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--games", type=int, default=4096, help="concurrent games (trees) per GPU")
    ap.add_argument("--sims", type=int, default=800, help="MCTS iterations per move")
    ap.add_argument("--net", default="mlp", choices=["mlp", "resnet"])
    ap.add_argument("--hidden", type=int, default=256)
    ap.add_argument("--graph-unroll", type=int, default=16)
    ap.add_argument("--leaves", type=int, default=4,
                    help="descents per tree and MCTS iteration (virtual loss; 1 = the strictly sequential search). "
                         "2 and 4 run as lane groups of the tree's warp (wave mode)")
    ap.add_argument("--torch-net", action="store_true",
                    help="evaluate the net with PyTorch/cuBLASLt GEMMs (4 launches) instead of the default: the "
                         "hand-written single-launch tcgen05 MLP kernel + programmatic dependent launch")
    ap.add_argument("--cpu-trees", type=int, default=256, help="trees of the CPU-baseline sample")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="CPU-baseline budget")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the env-kernel / INT32 side measurements")
    ap.add_argument("--scale-games", type=int, default=65536,
                    help="also report throughput at this many games/GPU (0 = skip); not the headline value")
    ap.add_argument("--no-iteration", action="store_true",
                    help="skip extra.iteration (BASELINE configs[4]: self-play + replay all-gather + training + weight "
                         "broadcast; the only part of the bench that moves bytes over NCCL)")
    ap.add_argument("--iteration-plies", type=int, default=70, help="lockstep plies of extra.iteration (a game lasts ~60)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm's timed steps")
    return args


# ------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled every 50 ms DURING the timed regions.  nvidia-smi takes 50-200 ms
    to deliver its first line, so it is started before the warm-up and every line is stamped on arrival; stop() keeps
    the lines that arrived inside the windows marked by window_begin() / window_end() (the timed regions)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.proc, self.lines = gpu_index, None, []
        self.windows, self._t0 = [], None

    def window_begin(self):
        self._t0 = time.monotonic()

    def window_end(self):
        if self._t0 is not None:
            self.windows.append((self._t0, time.monotonic()))
            self._t0 = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.monotonic(), line.strip()))

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        # a line describes the ~50 ms before it arrived: keep those that arrived inside a window (or just after it)
        inside = [ln for t, ln in self.lines if any(a <= t <= b + 0.06 for a, b in self.windows)]
        if not self.windows:
            inside = [ln for _, ln in self.lines]
        for ln in inside:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                pw.append(float(f[3]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------- CPU arm
def cpu_selfplay_sample(n_trees: int, n_sims: int, net_kind: str, hidden: int, budget_s: float, steps: int | None,
                        warmup: int = 1, leaves: int = 1):
    """The oracle port on the host cores: C sequential MCTS trees (oracle.c, OpenMP over trees)
    stepped in lockstep with the SAME policy/value net evaluated by PyTorch on the CPU in fp32.
    One step = one n_sims-iteration search from each of n_trees reachable roots."""
    import numpy as np
    import torch

    from betazero_b200 import net as netmod
    from oracle import pyoracle as po

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    po.set_num_threads(cores)  # torchrun exports OMP_NUM_THREADS=1
    net = netmod.make_net(net_kind, hidden=hidden, seed=0, device="cpu", dtype=torch.float32)
    me, opp = po.playout_boards(n_trees, seed=42)
    forest = po.OracleForest(n_trees, leaves=leaves)  # the same search definition as the GPU arm

    def one_step():
        forest.reset(me, opp)
        with torch.no_grad():
            for _ in range(n_sims // leaves):
                forest.select()
                logits, v = net(torch.from_numpy(forest.planes))
                w = torch.softmax(logits, dim=-1).numpy()
                forest.expand_backup(w, v.numpy())

    t0 = time.perf_counter()
    one_step()  # warm-up, also calibrates the step count to the budget
    t_one = time.perf_counter() - t0
    for _ in range(max(0, warmup - 1)):
        one_step()
    if steps is None:
        steps = max(1, min(50, int(budget_s / max(t_one, 1e-3))))
    t0 = time.perf_counter()
    for _ in range(steps):
        one_step()
    dt = time.perf_counter() - t0
    sims = steps * n_trees * n_sims
    return {"value": sims / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{steps} steps x {n_trees} trees x {n_sims} sims, {leaves} leaves per iteration (C oracle trees, "
                      f"OpenMP {po.num_threads()} threads, torch fp32 {net_kind} net on CPU, batch {n_trees * leaves}); {dt:.1f} s",
            "positions_per_sec": steps * n_trees / dt, "ms_per_step": 1e3 * dt / steps, "steps": steps}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # rank 0 alone runs the CPU arm
    # the same config object as the GPU arm prints for these arguments (the CPU arm itself evaluates the net with torch on
    # the host cores; `net_backend` names what the GPU arm uses)
    args.kernel_net = (not args.torch_net) and args.net == "mlp" and args.hidden == 256
    # W warm-up steps, then exactly K timed steps; one step = one search over the bounded sample
    r2 = cpu_selfplay_sample(args.cpu_trees, args.sims, args.net, args.hidden, 0, args.steps, args.warmup, args.leaves)
    line = {
        "impl": "reference", "metric": METRIC, "value": r2["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": r2["steps"], "warmup": args.warmup, "ms_per_step": r2["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
        # the same workload definition as the GPU arm, plus what this arm really timed: a bounded sample of its trees
        "config": dict(workload_config(args), trees_timed=args.cpu_trees,
                       timed_sample=f"{args.cpu_trees} of the {args.games} trees per step (bounded CPU sample)"),
        "cpu_baseline": {k: r2[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": r2["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "positions_per_sec": r2["positions_per_sec"], "gpu_launches": 0,
    }
    emit(line)


def kernel_net_label(rows):
    if rows <= 74 * 128:
        return ("bz_mlp_forward_pair (tcgen05 cta_group::2, weights resident in shared memory, one launch) "
                "+ programmatic dependent launch")
    return ("bz_mlp_forward_pair2 (tcgen05 cta_group::2, two ping-ponged 128-row tiles per CTA pair, one launch) "
            "+ programmatic dependent launch")


def search_label(leaves):
    if leaves <= 1:
        return "PUCT, one descent per tree and iteration (bit-exact vs oracle/mcts_ref.py MCTS.select)"
    return (f"PUCT, {leaves} descents per tree and iteration with virtual loss (north_star (b)); bit-exact vs "
            "oracle/mcts_ref.py MCTS.select_vl")


def workload_config(args):
    return {"workload": f"reversi8x8 self-play, {args.sims} sims/move, {args.games} games/GPU (BASELINE configs[3]), "
                        + (f"{args.leaves} virtual-loss descents per tree and iteration" if args.leaves > 1
                           else "one descent per tree and iteration"),
            "games_per_gpu": args.games, "trees_timed": args.games, "sims_per_move": args.sims, "leaves_per_iteration": args.leaves,
            "search": search_label(args.leaves),
            "evaluator": (f"policy/value MLP 128-{args.hidden}-{args.hidden}-{args.hidden}-(65+1), bf16, random init"
                          if args.net == "mlp" else f"policy/value {args.net} (hidden {args.hidden}), bf16, random init"),
            "net_backend": (("inside search_fused_kernel: tcgen05 cta_group::2 on CTA pairs, weight image resident in shared "
                             "memory for the whole move, leaf planes written from registers into the A operand")
                            if getattr(args, "one_launch", False) else
                            kernel_net_label(args.games * args.leaves) if getattr(args, "kernel_net", False)
                            else "PyTorch/cuBLASLt GEMMs"),
            "launches_per_move": (3 if getattr(args, "one_launch", False) else None),
            "l2_policy": "working set > L2: tree pools of one rank span GBs (no flush needed)",
            "sharding": f"games sharded over {args.gpus} GPU(s), no data-path collective"}


# ------------------------------------------------------------------------------------------- GPU arm
def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from betazero_b200 import env, mcts, selfplay
    from betazero_b200 import net as netmod

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device: the engine has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # stdout carries exactly one JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    B, S, K = args.games, args.sims, args.leaves
    if S % K:
        raise SystemExit("--sims must be a multiple of --leaves")
    net = netmod.make_net(args.net, hidden=args.hidden, seed=0)
    kernel_net = (not args.torch_net) and hasattr(net, "fused_kernel_ok") and net.fused_kernel_ok(
        torch.empty((1, 2, 8, 8), dtype=torch.bfloat16, device="cuda"))
    args.kernel_net = kernel_net
    if hasattr(net, "forward_raw"):
        evaluator = mcts.FusedNetEvaluator(net, use_kernel=None if kernel_net else False)
    else:
        evaluator = mcts.NetEvaluator(net)
    sp = selfplay.BatchedSelfPlay(B, S, evaluator, temp_plies=8, seed=1234, rank=rank, world=world,
                                  graph_unroll=args.graph_unroll, n_leaves=K)
    sp.prepare()
    args.one_launch = bool(sp.mcts.one_launch)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    roots_me = torch.empty((args.steps, B), dtype=torch.int64, device="cuda")  # the positions searched at every timed step
    roots_opp = torch.empty_like(roots_me)                                     # (the e2e region searches the same ones)
    for _ in range(args.warmup):
        roots_me[0].copy_(sp.me)  # the timed loop's own copies, so that nothing in it runs for the first time
        roots_opp[0].copy_(sp.opp)
        sp.play_move()
    barrier()

    # ---- timed region 1: device-resident self-play (value) ------------------------------------
    l0 = sp.total_launches()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    sampler.window_begin()
    ev0.record()
    for i in range(args.steps):
        roots_me[i].copy_(sp.me)
        roots_opp[i].copy_(sp.opp)
        sp.play_move()
    ev1.record()
    barrier()
    sampler.window_end()
    ms = ev0.elapsed_time(ev1)
    launches = sp.total_launches() - l0
    sp.mcts.check_errors()
    tstats = sp.mcts.stats()  # d and b of the last search
    if args.dump_outputs and rank == 0:
        dump_outputs(torch, sp, args.dump_outputs)  # before region 2, whose searches replace the trees

    # ---- timed region 2: end to end through the host-facing search API (e2e) ---------------------
    # per step: roots in pinned host memory -> H2D -> n_sims-iteration search -> pi + move -> D2H
    # (BatchedMCTS.search_host: the public call for boards that live in host memory -- it stages the roots in pinned memory,
    # copies them in, searches, copies pi and the move out and synchronises, every call)
    h_me = roots_me.cpu().pin_memory()    # the positions of the timed steps above, now in host memory
    h_opp = roots_opp.cpu().pin_memory()
    sp.mcts.search_host(h_me[0], h_opp[0], S)  # untimed: the first call captures the CUDA graph of the sequence
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    sampler.window_begin()
    e0.record()
    for i in range(args.steps):
        h_pi, h_act = sp.mcts.search_host(h_me[i], h_opp[i], S)  # returns after the stream synchronisation: the caller reads the result
    e1.record()
    barrier()
    sampler.window_end()
    ms_e2e = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None  # sampled over both timed regions (value and e2e)
    h2d = 2 * B * 8
    d2h = B * 65 * 4 + B

    # ---- the dominant kernel, timed launch by launch ------
    one_launch = bool(sp.mcts.one_launch)
    if one_launch:
        # search_fused_kernel: the whole search of a ply (tree kernels + net) is ONE launch
        step_kernel_ms, net_kernel_ms, probe_kind = probe_one_launch(torch, sp, S // K), None, \
            "CUDA events around each of 8 launches (one per ply) on the launching stream"
    else:
        # fused expand/backup + select + gather of one iteration
        step_kernel_ms, net_kernel_ms, probe_kind = probe_iteration_split(torch, sp, S // K - 1)

    # max over ranks, whole-job aggregate
    t = torch.tensor([ms, ms_e2e], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = float(t[0].item()), float(t[1].item())
    total_sims = world * args.steps * B * S
    value = total_sims / (ms * 1e-3)
    e2e_value = total_sims / (ms_e2e * 1e-3)

    peak = None
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak, peak_src = (peaks["hbm_gbs"], "measured") if "hbm_gbs" in peaks else (6650.0, "fallback")
        d = tstats["mean_depth"]
        bmean = tstats["edges"] / max(1, tstats["sims"])  # edges created per iteration ~ mean children of a new node
        bytes_per_sim = 28 * d + 12 * d * bmean + 13 * bmean + 312  # SURVEY.md 8d
        sims_per_launch = B * S if one_launch else B * K
        achieved = bytes_per_sim * sims_per_launch / (step_kernel_ms * 1e-3) / 1e9
        traffic, issue, static_note = None, None, None
        try:
            prof = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            if one_launch:
                same = B == 4096 and S == 800 and K == 4  # the configuration of the static capture
                traffic = prof.get("search_fused_dram_bytes_per_launch") if same else None
                winst = prof.get("search_fused_warp_inst_per_launch") if same else None
                static_note = prof.get("search_fused_note")
            else:
                traffic = prof.get("mcts_step_dram_bytes_per_launch" if K == 1 else f"mcts_step_wave{K}_dram_bytes_per_launch")
                winst = prof.get("mcts_step_warp_inst_per_launch" if K == 1 else f"mcts_step_wave{K}_warp_inst_per_launch")
            if winst and B == 4096:
                # second roofline of the same kernel: warp instructions issued (ncu count per launch at this batch) against
                # the issue rate of the chip, 148 SMs x 4 schedulers x 1 instruction/clk at the sampled SM clock
                clk = ((clocks or {}).get("sm_mhz") or 1965.0) * 1e6
                peak_issue = 148 * 4 * clk
                issue = {"bound": "issue", "warp_inst_per_launch": winst,
                         "warp_inst_source": "profiles/traffic.json (static: ncu smsp__inst_executed.sum of this kernel at "
                                             "this batch, not counted in this run)",
                         "achieved": winst / (step_kernel_ms * 1e-3) / 1e9,
                         "peak": peak_issue / 1e9, "unit": "G warp-inst/s", "frac": winst / (step_kernel_ms * 1e-3) / peak_issue}
        except Exception:
            pass
        # third view of the same kernel when it contains the net (the one-launch search): the MLP's useful flops (one
        # evaluation per simulation, 2 x (128 x 256 + 2 x 256 x 256 + 256 x 66) flop for the reference's architecture)
        # against the measured dense bf16 peak
        tensor_view = None
        if one_launch and args.net == "mlp" and args.hidden == 256:
            flop_per_leaf = 2 * (128 * 256 + 2 * 256 * 256 + 256 * 66)
            tf = flop_per_leaf * sims_per_launch / (step_kernel_ms * 1e-3) / 1e12
            tpeak = peaks.get("bf16_tflops_sustained") or peaks.get("bf16_tflops")
            tensor_view = {"bound": "tensor", "achieved": tf, "peak": tpeak, "unit": "TFLOP/s", "frac": (tf / tpeak) if tpeak else None,
                           "flop_per_simulation": flop_per_leaf,
                           "note": "useful MLP flops only (112 of the 128 rows of a tile are leaves; the head's 80-wide tile "
                                   "counts as 66); peak = MEASURED_PEAKS.json sustained dense bf16"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "fp32 tree statistics / u64 bitboards / bf16 net", "data": "synthetic",
            "config": workload_config(args),
            "positions_per_sec": world * args.steps * B / (ms * 1e-3),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": {"kernel": ("search_fused_kernel (one launch per move: K5 select + K6 gather + K7 expand/backup of all "
                                    f"{S // K} iterations, {K} leaves per tree, and the policy/value MLP on tcgen05 CTA pairs)"
                                    if one_launch else
                                    "step_kernel<reversi> (K7 expand/backup + K5 select + K6 gather)" if K == 1 else
                                    f"step_wave_kernel<reversi, {32 // K} lanes per descent> (K7 + K5 + K6, {K} leaves per tree)"),
                         "bound": "hbm",
                         "achieved": achieved, "peak": peak, "peak_source": peak_src, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic,
                         "traffic_source": "profiles/traffic.json (static: dram__bytes_read.sum + dram__bytes_write.sum of "
                                           "one ncu --set full capture of this kernel, not measured in this run)",
                         "kernel_ms": step_kernel_ms, "kernel_ms_probe": probe_kind,
                         "net_kernel_ms": net_kernel_ms,
                         "bytes_per_sim": bytes_per_sim, "mean_depth": d, "mean_children": bmean,
                         "sims_per_launch": sims_per_launch, "issue": issue, "tensor": tensor_view, "static_note": static_note},
            "tree": {"mean_depth": d, "edges_per_sim": bmean, "pool_bytes": sp.pools.nbytes()},
            "selfplay": sp.stats(),
        }
    else:
        line = None

    # ---- BASELINE configs[4]: one full AlphaZero iteration; EVERY rank takes part (replay all-gather + weight broadcast
    # over NCCL are the only collectives of the design), rank 0 reports
    pool_free = None
    if not args.no_iteration:
        del sp
        torch.cuda.empty_cache()
        pool_free = True
        it_line = iteration_block(args, rank, world)
        if rank == 0:
            line.setdefault("extra", {})["iteration"] = it_line

    if rank == 0:
        if not args.no_extra and world == 1:
            if not pool_free:
                del sp
                torch.cuda.empty_cache()
            ex = line.setdefault("extra", {})
            ex.update(side_measurements(torch, env, peak))
            if not args.no_cpu_baseline:
                ex["env_cpu_baseline"] = env_cpu_baseline(ex)
            if hasattr(net, "forward_raw"):
                ex["full_game"] = full_game(torch, mcts, selfplay, net, args)
                ex["tree_reuse"] = tree_reuse(torch, mcts, selfplay, net, args)
                ex["depth_sweep"] = depth_sweep(torch, mcts, selfplay, netmod, args)
                ex["config3_1024_trees_100_sims"] = config3(torch, mcts, selfplay, net, args)
                ex["other_net_backend"] = alt_backend(torch, mcts, selfplay, net, args)
                if one_launch:  # the same search through the per-iteration kernels (select / MLP / step, CUDA graph + PDL)
                    ex["per_iteration_kernels"] = alt_backend(torch, mcts, selfplay, net, args, same_backend=True,
                                                              one_launch=False, split=True)
                if K != 1:  # the strictly sequential search (one leaf per tree and iteration) on the same workload
                    ex["one_leaf_per_iteration"] = alt_backend(torch, mcts, selfplay, net, args, leaves=1, same_backend=True)
            if args.scale_games and args.scale_games != B:
                ex["at_scale"] = at_scale(torch, mcts, selfplay, net, args, args.scale_games, 1)
                if K != 1:
                    ex["at_scale_virtual_loss"] = [at_scale(torch, mcts, selfplay, net, args, g, K)
                                                   for g in sorted({16384, args.scale_games}) if g != B]
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = {k: v for k, v in cpu_selfplay_sample(
                args.cpu_trees, S, args.net, args.hidden, args.cpu_seconds, None, leaves=K).items()
                if k in ("value", "unit", "cores", "kind", "sample")}
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def dump_outputs(torch, sp, out_dir, budget=64 << 20):
    """What a caller of the timed step (BatchedSelfPlay.play_move) has after its last call, one row per game, as float32
    DIR/<name>.npy: the root statistics of that move's search (root_visits, root_pi = the visit distribution recorded for
    training, root_q), the move played (action, 64 = pass) and the position the game stands at afterwards (board: +1 the
    side to move, -1 its opponent, cell = row * 8 + col; player; ply).  Rows beyond `budget` bytes: a fixed, seeded
    sample of the games, their indices in rows.npy.  counters.npy (float64): the self-play counters of BatchedSelfPlay.stats."""
    import numpy as np

    B = sp.n_games
    counts, pi, q = sp.mcts.root_policy()
    bits = torch.arange(64, device=sp.me.device)

    def cells(b):
        return ((b[:B, None] >> bits) & 1).float()

    out = {"root_visits": counts[:B].float(), "root_pi": pi[:B], "root_q": q[:B], "action": sp.last_action[:B].float(),
           "board": cells(sp.me) - cells(sp.opp), "player": sp.player[:B].float(), "ply": sp.ply[:B].float()}
    out = {k: v.cpu().numpy().astype(np.float32) for k, v in out.items()}
    row_bytes = sum(v[0].nbytes for v in out.values()) + 8  # + its index in rows.npy
    room = budget - 4096  # .npy headers and counters.npy
    if B * row_bytes > room:
        rows = np.sort(np.random.default_rng(0).choice(B, room // row_bytes, replace=False))
        out = {k: v[rows] for k, v in out.items()}
        out["rows"] = rows.astype(np.float64)
    out["counters"] = sp.counters.cpu().numpy().astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def iteration_block(args, rank, world):
    """extra.iteration: betazero_b200.loop.run_iteration at the bench's configuration (mirrors the reference's training
    loop, SL/train.py:85-113, behind batched self-play).  Per-phase device times, gathered bytes, NCCL bus bandwidth."""
    from betazero_b200 import loop

    try:
        la = loop.default_args(games=args.games, sims=args.sims, leaves=args.leaves, plies=args.iteration_plies,
                               net=args.net, hidden=args.hidden, seed=1234)
        st = loop.LoopState(la, rank, world)
        # two iterations, the second is reported: the first one also pays the one-time costs of the phases that run once
        # per iteration (cuBLAS / optimiser / sort kernels loading, NCCL channel set-up, allocator growth)
        first = loop.run_iteration(st, 0)
        out = loop.run_iteration(st, 1)
        out["first_iteration_ms"] = first["ms"]
        out["what"] = ("BASELINE configs[4]: lockstep self-play from the start positions (slots recycle as games end) -> "
                       "replay drain + NCCL all-gather (one packed buffer) -> Adam steps on augmented batches -> "
                       "NCCL weight broadcast + in-place refresh of the search's weight image")
        del st
        import torch

        torch.cuda.empty_cache()
        return out
    except Exception as e:
        if world > 1:
            raise  # a rank that skipped a collective would hang the others: fail loudly instead
        return {"error": f"{type(e).__name__}: {e}"}


def probe_iteration_split(torch, sp, n_iter):
    """Mean duration of the tree kernel and of the evaluator inside an MCTS iteration, over the deep-tree half of one search.
    Preferred: CUDA events recorded INSIDE a replayed graph (event-record nodes, torch `external=True`): 16 iterations of
    [net, event, tree kernel, event] -- an interval holds the kernel and the dependency latency of its graph edges, not
    an eager launch.  Fallback: eager launches behind a busy GPU.  Returns (tree_ms, net_ms or None, probe description)."""
    try:
        pairs = [(torch.cuda.Event(enable_timing=True, external=True), torch.cuda.Event(enable_timing=True, external=True))
                 for _ in range(16)]
        sp.mcts.reset(sp.me, sp.opp)
        sp.mcts.select()
        for _ in range(2):  # warm-up of the exact sequence that is captured
            sp.mcts.evaluate()
            sp.mcts.step()
        pg = torch.cuda.CUDAGraph()
        with torch.cuda.graph(pg):
            for a, b in pairs:
                sp.mcts.evaluate()
                a.record()
                sp.mcts.step()
                b.record()
        sp.mcts.reset(sp.me, sp.opp)
        sp.mcts.select()
        k_ms, n_ms = [], []
        done = 0
        while done + 16 <= n_iter:
            pg.replay()
            done += 16
            if done * 2 >= n_iter:  # deep-tree half
                torch.cuda.synchronize()
                k_ms += [a.elapsed_time(b) for a, b in pairs]
                n_ms += [pairs[i][1].elapsed_time(pairs[i + 1][0]) for i in range(15)]
        torch.cuda.synchronize()
        if k_ms:
            return sum(k_ms) / len(k_ms), sum(n_ms) / len(n_ms), "events inside a replayed CUDA graph"
    except Exception as e:  # older torch without external events, or capture refused: fall back
        print(f"graph-event probe unavailable ({type(e).__name__}: {e}); using eager launches", file=sys.stderr)
    sp.mcts.reset(sp.me, sp.opp)
    sp.mcts.select()
    evs = []
    n_probe = min(n_iter, 400)
    for i in range(n_probe):
        sp.mcts.evaluate()
        # keep the GPU busy while the CPU enqueues the probed launch, so [a, b] holds the kernel only
        # (eager launches are CPU-bound; without this the interval would include a launch gap)
        torch.cuda._sleep(60_000)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        sp.mcts.step()
        b.record()
        evs.append((a, b))
    torch.cuda.synchronize()
    k_ms = [a.elapsed_time(b) for a, b in evs]
    half = k_ms[len(k_ms) // 2:] or [0.0]  # deep-tree half
    return sum(half) / len(half), None, "eager launches behind a busy GPU (includes ~4 us of launch latency)"



def probe_one_launch(torch, sp, n_iter, plies=8):
    """Mean duration of search_fused_kernel (one launch = the whole search of a ply) over `plies` searches of the current
    positions, CUDA events on the launching stream right around the launch."""
    evs = []
    for _ in range(plies):
        sp.mcts.reset(sp.me, sp.opp)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        sp.mcts.search_one_launch(n_iter)
        b.record()
        evs.append((a, b))
    torch.cuda.synchronize()
    return sum(a.elapsed_time(b) for a, b in evs) / len(evs)


def alt_backend(torch, mcts, selfplay, net, args, leaves=None, same_backend=False, one_launch=None, split=False):
    """The headline workload with the OTHER net backend (library GEMMs if the headline used the tcgen05 MLP
    kernel, and vice versa), or with another number of leaves per iteration, so one bench line shows both."""
    from betazero_b200 import _lib as bzlib

    leaves = args.leaves if leaves is None else leaves
    use_kernel = getattr(args, "kernel_net", False) if same_backend else not getattr(args, "kernel_net", False)
    try:
        ev = mcts.FusedNetEvaluator(net, use_kernel=None if use_kernel else False)
        sp = selfplay.BatchedSelfPlay(args.games, args.sims, ev, temp_plies=8, seed=1234, graph_unroll=args.graph_unroll,
                                      n_leaves=leaves, one_launch=one_launch)
        sp.prepare()
        for _ in range(3):
            sp.play_move()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        n = 10
        for _ in range(n):
            sp.play_move()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n
        sp.mcts.check_errors()
        out = {"sims_per_sec": args.games * args.sims / (ms * 1e-3), "ms_per_step": ms, "leaves_per_iteration": leaves,
               "search": search_label(leaves), "one_launch": bool(sp.mcts.one_launch),
               "net_backend": kernel_net_label(args.games * leaves) if use_kernel else "PyTorch/cuBLASLt GEMMs"}
        if split:
            tree_ms, net_ms, probe = probe_iteration_split(torch, sp, args.sims // leaves - 1)
            out["per_iteration"] = {"tree_kernel_ms": tree_ms, "net_kernel_ms": net_ms, "probe": probe}
        return out
    except Exception as e:
        return {"error": f"{type(e).__name__}: {e}"}
    finally:
        bzlib.set_pdl(False)


def _timed_plies(torch, sp, warm, n):
    for _ in range(warm):
        sp.play_move()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        sp.play_move()
    e1.record()
    torch.cuda.synchronize()
    sp.mcts.check_errors()
    return e0.elapsed_time(e1) / n


def at_scale(torch, mcts, selfplay, net, args, games, leaves):
    """Same loop with many more concurrent games (the north-star asks for >= 4096 per GPU): with one leaf per iteration the
    tree kernel switches to 8-lane groups (4 trees per warp); with virtual loss it stays in wave mode (a warp per tree)."""
    G, S = games, args.sims
    try:
        evaluator = mcts.FusedNetEvaluator(net) if hasattr(net, "forward_raw") else mcts.NetEvaluator(net)
        sp = selfplay.BatchedSelfPlay(G, S, evaluator, temp_plies=8, seed=99, graph_unroll=args.graph_unroll, n_leaves=leaves)
        sp.prepare()
        ms = _timed_plies(torch, sp, 2, 3)
        st = sp.mcts.stats()
        d, b = st["mean_depth"], st["edges"] / max(1, st["sims"])
        lanes = 32 // leaves if leaves in (2, 4) else (8 if G >= 32768 else (16 if G >= 8192 else 32))
        return {"games_per_gpu": G, "sims_per_sec": G * S / (ms * 1e-3), "positions_per_sec": G / (ms * 1e-3),
                "ms_per_step": ms, "lanes_per_descent": lanes, "leaves_per_iteration": leaves, "mean_depth": d,
                "mean_children": b, "pool_bytes": sp.pools.nbytes(), "one_launch": bool(sp.mcts.one_launch),
                "launches_per_move": (2 + -(-G // sp.mcts.ONE_LAUNCH_MAX_TREES)) if sp.mcts.one_launch else None}
    except Exception as e:  # never let the side measurement break the headline line
        return {"games_per_gpu": G, "leaves_per_iteration": leaves, "error": f"{type(e).__name__}: {e}"}
    finally:
        from betazero_b200 import _lib as bzlib

        bzlib.set_pdl(False)


def tree_reuse(torch, mcts, selfplay, net, args, plies=40):
    """Opt-in tree reuse (bz_mcts_reroot): every move's search continues on the subtree of the move played, so a move's
    root carries the kept visits plus sims/move new ones and the trees go deeper.  Reported: the same sims/s metric (new
    simulations only), the re-rooting kernel's share of a ply, the root visit totals and the tree depth."""
    B, S, K = args.games, args.sims, args.leaves
    try:
        ev = mcts.FusedNetEvaluator(net, use_kernel=None if getattr(args, "kernel_net", False) else False)
        sp = selfplay.BatchedSelfPlay(B, S, ev, temp_plies=8, seed=4321, graph_unroll=args.graph_unroll, n_leaves=K, reuse=True)
        sp.prepare()
        for _ in range(4):
            sp.play_move()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(plies):
            sp.play_move()
        e1.record()
        torch.cuda.synchronize()
        sp.mcts.check_errors()
        ms = e0.elapsed_time(e1) / plies
        st = sp.mcts.stats()
        inherited = float(sp.pools.inherited.float().mean().item())
        root_visits = float(sp.pools.sim_count.float().mean().item())
        units = float(sp.pools.arena_used.float().mean().item())
        # the re-rooting kernel alone, on the trees as they stand (same move twice is not possible: time one call)
        sp.search()
        sp.advance()
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r0.record()
        sp.mcts.advance(sp.last_action, sp.me, sp.opp)
        r1.record()
        torch.cuda.synchronize()
        return {"plies": plies, "games_per_gpu": B, "leaves_per_iteration": K, "ms_per_ply": ms,
                "sims_per_sec": B * S / (ms * 1e-3), "reroot_kernel_ms": r0.elapsed_time(r1),
                "mean_root_visits_after_search": root_visits, "mean_inherited_visits": inherited,
                "mean_depth": st["mean_depth"], "mean_arena_units_used": units, "arena_units": sp.pools.arena_units,
                "pool_bytes": sp.pools.nbytes() + sp.pools.scratch.numel() * 4,
                "note": "sims/s counts the NEW simulations of a move only; off by default (the goldens pin a fresh tree per move)"}
    except Exception as e:
        return {"error": f"{type(e).__name__}: {e}"}
    finally:
        from betazero_b200 import _lib as bzlib

        bzlib.set_pdl(False)


def full_game(torch, mcts, selfplay, net, args, plies=80, bucket=10):
    """Whole games instead of the opening plies of the headline region: `plies` lockstep plies from the start position
    (a Reversi game lasts ~60, so every slot finishes a game and restarts: slot recycling, replay flushes and the late-game
    small trees are all inside the timed region).  Throughput over the whole run and per bucket of plies, with the tree
    depth of the last search of each bucket."""
    B, S, K = args.games, args.sims, args.leaves
    try:
        ev = mcts.FusedNetEvaluator(net, use_kernel=None if getattr(args, "kernel_net", False) else False)
        sp = selfplay.BatchedSelfPlay(B, S, ev, temp_plies=8, seed=4321, graph_unroll=args.graph_unroll, n_leaves=K)
        sp.prepare()
        marks = [torch.cuda.Event(enable_timing=True) for _ in range(plies // bucket + 1)]
        depth = []
        torch.cuda.synchronize()
        marks[0].record()
        for i in range(plies // bucket):
            for _ in range(bucket):
                sp.play_move()
            marks[i + 1].record()
            st = sp.mcts.stats()  # tiny D2H read between buckets (inside the timed run)
            depth.append(st["mean_depth"])
        torch.cuda.synchronize()
        sp.mcts.check_errors()
        n = (plies // bucket) * bucket
        total_ms = marks[0].elapsed_time(marks[-1])
        per = [marks[i].elapsed_time(marks[i + 1]) / bucket for i in range(plies // bucket)]
        stats = sp.stats()
        return {"plies": n, "games_per_gpu": B, "leaves_per_iteration": K, "ms_per_ply": total_ms / n,
                "sims_per_sec": B * S * n / (total_ms * 1e-3), "positions_per_sec": B * n / (total_ms * 1e-3),
                "games_finished": stats["games"], "replay_records": stats["replay_records"], "dropped": stats["dropped"],
                "ply_buckets": [{"plies": f"{i * bucket}-{(i + 1) * bucket - 1}", "ms_per_ply": per[i],
                                 "sims_per_sec": B * S / (per[i] * 1e-3), "mean_depth_last_search": depth[i]}
                                for i in range(plies // bucket)],
                "note": "sims counted as games x sims/move for every ply; slots whose game just ended search the start position"}
    except Exception as e:
        return {"error": f"{type(e).__name__}: {e}"}
    finally:
        from betazero_b200 import _lib as bzlib

        bzlib.set_pdl(False)


def depth_sweep(torch, mcts, selfplay, netmod, args, scales=(1, 32, 128, 512)):
    """Depth sensitivity: a random-init net has nearly flat priors, so its trees stay shallow (depth ~3).  A trained net has
    peaked priors.  Multiplying the policy head by `scale` sharpens the priors of the SAME net; the search then goes
    deeper and every extra tree level adds one dependent load round per descent.  Reports sims/s against mean depth."""
    B, S, K = args.games, args.sims, args.leaves
    out = []
    try:
        for scale in scales:
            net = netmod.make_net(args.net, hidden=args.hidden, seed=0)
            with torch.no_grad():
                net.policy.weight.mul_(scale)
                net.policy.bias.mul_(scale)
            ev = mcts.FusedNetEvaluator(net, use_kernel=None if getattr(args, "kernel_net", False) else False)
            sp = selfplay.BatchedSelfPlay(B, S, ev, temp_plies=8, seed=1234, graph_unroll=args.graph_unroll, n_leaves=K)
            sp.prepare()
            ms = _timed_plies(torch, sp, 6, 6)  # plies 6..11: mid-opening positions with ~8-10 legal moves
            st = sp.mcts.stats()
            out.append({"policy_logit_scale": scale, "mean_depth": st["mean_depth"],
                        "mean_children": st["edges"] / max(1, st["sims"]), "ms_per_step": ms,
                        "sims_per_sec": B * S / (ms * 1e-3)})
            del sp, ev, net
            torch.cuda.empty_cache()
        return out
    except Exception as e:
        return out + [{"error": f"{type(e).__name__}: {e}"}]
    finally:
        from betazero_b200 import _lib as bzlib

        bzlib.set_pdl(False)


def config3(torch, mcts, selfplay, net, args, games=1024, sims=100, plies=70):
    """BASELINE configs[2] / SURVEY 8d "Config 3": 1024 concurrent trees, 100 sims/move, random-init bf16 net, full games
    from the start position; sims/s, positions/s and the time split env / tree (+ gather, fused into it) / net."""
    K = args.leaves if sims % args.leaves == 0 else 1
    try:
        ev = mcts.FusedNetEvaluator(net, use_kernel=None if getattr(args, "kernel_net", False) else False)
        sp = selfplay.BatchedSelfPlay(games, sims, ev, temp_plies=8, seed=3, graph_unroll=8, n_leaves=K)
        sp.prepare()
        ms = _timed_plies(torch, sp, 3, plies)
        stats = sp.stats()
        tree_ms, net_ms, probe = probe_iteration_split(torch, sp, sims // K - 1)
        evs = []
        for _ in range(20):  # the move / terminal / replay kernel of a ply, behind a busy GPU (no launch gap inside)
            sp.search()
            torch.cuda._sleep(60_000)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            sp.advance()
            b.record()
            evs.append((a, b))
        torch.cuda.synchronize()
        env_ms = sum(a.elapsed_time(b) for a, b in evs) / len(evs)
        iters = sims // K
        return {"games": games, "sims_per_move": sims, "leaves_per_iteration": K, "plies": plies, "ms_per_ply": ms,
                "sims_per_sec": games * sims / (ms * 1e-3), "positions_per_sec": games / (ms * 1e-3),
                "games_finished": stats["games"],
                "split_ms_per_ply": {"tree_select_expand_backup_gather": None if tree_ms is None else tree_ms * iters,
                                     "net": None if net_ms is None else net_ms * iters,
                                     "env_move_terminal_replay": env_ms,
                                     "per_iteration": {"tree_kernel_ms": tree_ms, "net_kernel_ms": net_ms, "iterations": iters},
                                     "probe": probe + "; env: events around bz_selfplay_advance behind a busy GPU"}}
    except Exception as e:
        return {"error": f"{type(e).__name__}: {e}"}
    finally:
        from betazero_b200 import _lib as bzlib

        bzlib.set_pdl(False)


def env_cpu_baseline(extra, budget_boards=1 << 18):
    """SURVEY 8d / BASELINE.md 4.1: the reference-style env on the host cores beside K1 / K2 -- the oracle port of
    generate_possible_moves (64 x is_valid_move ray walks, reversi_board.py:25-41,87-88) and make_move (:43-59) on set A
    (synthetic) and set B (reachable, random playouts) boards, one thread and all cores."""
    import numpy as np

    from oracle import pyoracle as po

    cores = os.cpu_count() or 1
    out = {"kind": "port", "cores": cores,
           "what": "oracle.c grid + ray-walk restatement of ReversiBoard.generate_possible_moves + make_move (first legal move), "
                   "OpenMP over boards"}
    sets = {"set_a_synthetic": po.synthetic_boards(budget_boards, seed=0),
            "set_b_playouts": po.playout_boards(budget_boards // 8, seed=0)}
    try:
        for name, (me, opp) in sets.items():
            res = {"boards": int(me.size)}
            for label, nt in (("1_thread", 1), (f"{cores}_threads", cores)):
                po.set_num_threads(nt)
                po.legal_mask(me[:1024], opp[:1024])  # warm-up
                t0 = time.perf_counter()
                mask = po.legal_mask(me, opp)
                t1 = time.perf_counter()
                low = mask & (~mask + np.uint64(1))
                act = np.where(mask != 0, np.log2(np.maximum(low, 1).astype(np.float64)).astype(np.uint8), 64).astype(np.uint8)
                t2 = time.perf_counter()
                po.apply(me, opp, act)
                t3 = time.perf_counter()
                res[label] = {"legal_mask_boards_per_sec": me.size / (t1 - t0),
                              "mask_plus_apply_boards_per_sec": me.size / ((t1 - t0) + (t3 - t2))}
            out[name] = res
        po.set_num_threads(cores)
        k1 = extra.get("env_legal_mask", {}).get("boards_per_sec")
        k12 = extra.get("env_step_first_legal", {}).get("boards_per_sec")
        a = out["set_a_synthetic"][f"{cores}_threads"]
        if k1 and k12:
            out["gpu_over_cpu_all_cores"] = {"legal_mask": k1 / a["legal_mask_boards_per_sec"],
                                             "mask_plus_apply": k12 / a["mask_plus_apply_boards_per_sec"]}
        return out
    except Exception as e:
        out["error"] = f"{type(e).__name__}: {e}"
        return out


def side_measurements(torch, env, hbm_peak):
    """Config-2 env kernels at 2^26 boards (working set > L2) and the INT32 issue-rate microbench."""
    out = {}
    n = 1 << 26
    g = torch.Generator(device="cuda").manual_seed(0)
    a = torch.randint(-(2 ** 63), 2 ** 63 - 1, (n,), dtype=torch.int64, device="cuda", generator=g)
    b = torch.randint(-(2 ** 63), 2 ** 63 - 1, (n,), dtype=torch.int64, device="cuda", generator=g)
    c = torch.randint(-(2 ** 63), 2 ** 63 - 1, (n,), dtype=torch.int64, device="cuda", generator=g)
    me, opp = a & b, ~a & c
    del a, b, c
    mask = torch.empty_like(me)
    outs = (torch.empty_like(me), torch.empty(n, dtype=torch.uint8, device="cuda"), torch.empty_like(me), torch.empty_like(me))

    def timed(fn, reps=5):
        for _ in range(3):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    t1 = timed(lambda: env.legal_mask(me, opp, out=mask))
    t2 = timed(lambda: env.step_first_legal(me, opp, out=outs))
    out["env_legal_mask"] = {"boards": n, "ms": t1, "boards_per_sec": n / t1 * 1e3, "GBps": 24 * n / t1 / 1e6,
                             "hbm_frac": 24 * n / t1 / 1e6 / hbm_peak}
    out["env_step_first_legal"] = {"boards": n, "ms": t2, "boards_per_sec": n / t2 * 1e3, "GBps": 41 * n / t2 / 1e6,
                                   "hbm_frac": 41 * n / t2 / 1e6 / hbm_peak}
    blocks, threads, iters = 148 * 8, 256, 2048
    ops = env.int32_microbench(blocks, threads, iters)
    t3 = timed(lambda: env.int32_microbench(blocks, threads, iters), reps=3)
    peak_int = ops / t3 * 1e3
    out["int32_peak"] = {"alu_pipe_thread_inst_per_sec": peak_int, "ms": t3,
                         "note": "SHF+LOP3 mix (every instruction on the ALU pipe), 8 independent chains/thread, 148x8 CTAs x "
                                 "256 threads; counted in thread-instructions, the unit of the fractions below"}
    # INT32 roofline fraction, numerator and denominator both in ALU-pipe thread-instructions per second:
    #   frac = boards/s (this run) x ALU-pipe instructions per board (static property of the binary) / ALU-pipe peak (this run)
    inst = {}
    try:
        inst = json.load(open(os.path.join(ROOT, "profiles", "env_inst.json")))["kernels"]
    except Exception:
        pass
    for key, kern in (("env_legal_mask", "legal_mask_kernel"), ("env_step_first_legal", "step_first_legal_kernel")):
        k = inst.get(kern)
        if not k:
            continue
        per_board = k.get("ncu_alu_pipe_inst_per_board") or k["alu_pipe_inst_per_board"]
        rate = out[key]["boards_per_sec"] * per_board
        out[key]["roofline"] = {"bound": "int32 ALU pipe", "frac": rate / peak_int, "unit": "ALU-pipe thread-inst/s",
                                "achieved": rate, "peak": peak_int,
                                "alu_pipe_inst_per_board": per_board,
                                "alu_pipe_inst_per_board_source": "profiles/env_inst.json (static: executed ALU-pipe instructions "
                                                                  "per board from the ncu capture r1_env_kernels_raw.csv; "
                                                                  f"static SASS count {k['alu_pipe_inst_per_board']})",
                                "frac_computed_from": "boards/s of this run x static instructions per board / ALU-pipe peak of "
                                                      "this run"}
    return out


_REAL_STDOUT = None


def emit(line: dict) -> None:
    """The ONE JSON line of this run, written to the real stdout (see main)."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    args = parse()
    # Libraries (NCCL's version banner, torchrun notices, ...) print to fd 1; the contract is exactly one JSON
    # line on stdout, so fd 1 is pointed at stderr for the whole run and the result goes to the saved descriptor.
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
