"""One full AlphaZero iteration (BASELINE configs[4]): lockstep self-play on every GPU -> replay
gather (NCCL all-gather) -> training steps on the gathered records -> weight broadcast.

    torchrun --nproc-per-node 8 -m betazero_b200.loop --games 4096 --sims 800 --plies 70 --train-steps 8

Self-play is the hot path (hand-written kernels, no collective); the two collectives run once per
iteration (`dist.gather_replay`, `dist.broadcast_weights`).  Every rank trains on the same gathered
batch order with the same seed, so the replicas stay bit-identical and the broadcast is a
consistency guarantee rather than a necessity; with ``--train-on-rank0`` only rank 0 trains.
The training loop mirrors the reference's (Adam + cross-entropy, src/tic_tac_toe/SL/train.py:85-113) and, like it,
saves the model at the end (:204-214) -- here a state_dict checkpoint per iteration (``--checkpoint``; one file per
iteration when the path contains ``{iteration}``), resumable (``--resume``).  Prints one JSON line per iteration on rank 0.  With ``--eval-games N`` rank 0 also plays N games between the
trained net and the net before training (``match.BatchedMatch``) and adds their score and Elo to the line; with
``--eval-minimax DEPTH`` as well, it plays N more games between the trained net and the reference's minimax player of that
depth (``tournament.Minimax``) and adds them as ``eval_minimax``: a yardstick that stays the same across iterations.
With ``--eval-endgame EMPTIES`` rank 0 scores the trained net's moves on a fixed suite of 4096 positions with that many
empty squares against the exact solver (``betazero_b200.endgame``), at 0 simulations and at ``--sims`` / ``--leaves``, and
adds ``eval_endgame``; the suite is drawn and solved once per run.  With ``--endgame-empties E`` self-play hands every game to
the exact solver once a searched move leaves at most E empty squares, and runs a solver phase every ``--endgame-every``
plies (``selfplay.BatchedSelfPlay``); the line then has an ``endgame`` entry with the solver's counts and the time of its
phases.  ``--endgame-solve wld`` runs the win/draw/loss solver for both instead of the exact one (cheaper; the handover's
pi is then uniform over the moves that keep the result, and ``eval_endgame`` reports ``wld_accuracy`` only); both
entries name the solver.  With ``--resign V`` a self-play game that is not audited resigns at its first searched ply whose
q (W / N of the most visited root edge) is below V (-1: audit only); ``--resign-audit F`` games never resign and measure
the false positives, and ``--resign-fp P`` sets the next iteration's threshold from this iteration's gathered audited
games (``resign.calibrate``: the same on every rank, since every rank gathers the same replay).  The line then has a
``resign`` entry, and the checkpoint's ``extra`` holds the next threshold, which ``--resume`` restores.  With
``--fast-sims N`` a fraction ``--full-fraction P`` of the self-play plies (a Philox draw per ply) is searched with
``--sims`` and every other ply with N simulations (randomized search budgets); training batches are drawn from the full
plies' records only, after the resignation calibration, which uses every record.  The line then has a ``cap`` entry,
and the checkpoint's ``extra`` holds both settings.
"""
from __future__ import annotations

import argparse
import copy
import json
import os
import time
import warnings
from types import SimpleNamespace

import torch

from . import dist as bzd
from . import endgame, match, mcts, minimax, net, resign, selfplay, train


def default_args(**over) -> SimpleNamespace:
    """the command line's defaults as a namespace (for callers that drive iterations from Python: bench.py, tests)"""
    a = SimpleNamespace(games=4096, sims=800, leaves=4, plies=70, size=8, iterations=1, train_steps=8, batch=4096, lr=1e-4,
                        temp_plies=8, net="mlp", hidden=256, seed=0, train_on_rank0=False, checkpoint=None, resume=None,
                        reuse=False, eval_games=0, eval_minimax=None, eval_endgame=None, endgame_empties=0, endgame_every=8,
                        endgame_solve="exact", resign=None, resign_audit=0.1, resign_fp=None, fast_sims=None,
                        full_fraction=0.25)
    for k, v in over.items():
        if not hasattr(a, k):
            raise TypeError(f"unknown loop argument {k!r}")
        setattr(a, k, v)
    return a


ENDGAME_POSITIONS = 4096  # --eval-endgame: one launch of the one-launch search


class LoopState:
    """Everything one rank keeps across iterations: the bf16 inference net inside the search, the fp32 master copy and
    its optimiser, and the lockstep self-play driver."""

    def __init__(self, args, rank: int, world: int):
        self.args, self.rank, self.world = args, rank, world
        eg = int(getattr(args, "eval_games", 0))
        if eg < 0 or eg % 2:
            raise ValueError(f"eval_games must be an even number >= 0 (games are played in pairs); got {eg}")
        em = getattr(args, "eval_minimax", None)
        if em is not None:
            minimax.check_depth(em)
            if eg == 0:
                raise ValueError("eval_minimax plays --eval-games games: set eval_games > 0")
        solve = selfplay.check_endgame_solve(getattr(args, "endgame_solve", "exact"))
        self.endgame_suite = None  # --eval-endgame: drawn and solved once per run (rank 0)
        ee = getattr(args, "eval_endgame", None)
        if ee is not None:
            if not 1 <= int(ee) <= minimax.SOLVE_MAX_EMPTIES:
                raise ValueError(f"eval_endgame must be in 1 .. {minimax.SOLVE_MAX_EMPTIES} empty squares; got {ee}")
            if rank == 0:
                self.endgame_suite = endgame.positions(ENDGAME_POSITIONS, int(ee), args.size, args.seed)
                self.endgame_suite.wld = solve == "wld"
                endgame.solve_suite(self.endgame_suite)
        self.model = net.make_net(args.net, hidden=args.hidden, seed=args.seed)
        self.master = net.make_net(args.net, hidden=args.hidden, seed=args.seed, dtype=torch.float32)  # fp32 master weights
        self.opt = torch.optim.Adam(self.master.parameters(), lr=args.lr)  # the reference's optimiser family (SL/train.py:87)
        # resignation: --resign V, or -1 (audit only) when only --resign-fp is given; None = off
        threshold, fp = getattr(args, "resign", None), getattr(args, "resign_fp", None)
        if fp is not None and not float(fp) >= 0.0:
            raise ValueError(f"resign_fp must be a false-positive rate >= 0; got {fp}")
        if threshold is None and fp is not None:
            threshold = -1.0
        if threshold is not None:
            threshold = resign.check_threshold(threshold)
        self.first_iteration = 0
        if args.resume:
            self.first_iteration = train.load_checkpoint(args.resume, self.master, self.opt)
            self._publish()
            kept = torch.load(args.resume, map_location="cpu", weights_only=True).get("extra", {}).get("resign_threshold")
            if threshold is not None and kept is not None:
                threshold = resign.check_threshold(kept)
        self.evaluator = (mcts.FusedNetEvaluator(self.model) if hasattr(self.model, "forward_raw")
                          else mcts.NetEvaluator(self.model))
        self.sp = selfplay.BatchedSelfPlay(args.games, args.sims, self.evaluator, board_size=args.size,
                                           temp_plies=args.temp_plies, seed=args.seed, rank=rank, world=world,
                                           n_leaves=args.leaves, reuse=bool(getattr(args, "reuse", False)),
                                           graph_unroll=min(16, max(1, args.sims // args.leaves - 1)),
                                           endgame_empties=int(getattr(args, "endgame_empties", 0)),
                                           endgame_every=int(getattr(args, "endgame_every", 8)), endgame_solve=solve,
                                           resign_threshold=threshold, resign_audit=float(getattr(args, "resign_audit", 0.1)),
                                           fast_sims=getattr(args, "fast_sims", None),
                                           full_fraction=float(getattr(args, "full_fraction", 0.25)))
        self.sp.prepare()

    @torch.no_grad()
    def _publish(self) -> None:
        """master (fp32) -> inference net (bf16), in place: the captured CUDA graph keeps its pointers"""
        for dst, src in zip(self.model.parameters(), self.master.parameters()):
            dst.copy_(src)
        for dst, src in zip(self.model.buffers(), self.master.buffers()):
            dst.copy_(src)


def checkpoint_path(pattern: str, it: int) -> str:
    """``--checkpoint`` with ``{iteration}`` replaced by the iteration number: one file per iteration, kept for a
    tournament between them (``betazero_b200.tournament``).  Without the placeholder every iteration overwrites one file."""
    return pattern.replace("{iteration}", str(it))


def run_iteration(st: LoopState, it: int) -> dict:
    """self-play -> replay all-gather -> training steps -> weight broadcast; phases timed with CUDA events"""
    args, rank, world, sp = st.args, st.rank, st.world, st.sp
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
    torch.cuda.synchronize()
    eg_ms0, eg_stats0 = (sp.endgame_ms(), sp.stats()) if sp.eg is not None else (0.0, None)
    rs_stats0, rs_threshold = (sp.stats(), sp.resign_threshold) if sp.rs is not None else (None, None)
    cap_stats0 = sp.stats() if sp.cs is not None else None
    t0 = time.perf_counter()
    ev[0].record()
    for _ in range(args.plies):
        sp.play_move()
    ev[1].record()
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        shard = sp.drain_replay()
    replay = bzd.gather_replay(shard)
    gather_info = dict(bzd.last_gather)
    ev[2].record()
    n = replay["me"].shape[0]
    resign_line = None
    if sp.rs is not None:
        # the audited games of the gathered replay: every rank holds the same records, so every rank computes the same
        # false-positive rate and the same next threshold
        recs = resign.with_audit(replay, args.seed, sp.resign_audit)
        fp_target = getattr(args, "resign_fp", None)
        if fp_target is not None:
            sp.set_resign_threshold(resign.calibrate(recs, float(fp_target), keep=rs_threshold))
        n_games = int(torch.unique(replay["game"]).numel()) if n else 0
        resign_line = {"threshold": rs_threshold, "next_threshold": sp.resign_threshold, "audit": sp.resign_audit,
                       "fp_target": fp_target, "fp": resign.false_positive_rate(recs, rs_threshold),
                       "audited_games": resign.audited_games(recs), "plies_per_game": n / n_games if n_games else None}
    # randomized budgets: the policy targets of fast plies come from cheap searches, so the batches are drawn from the
    # full records only (after the calibration above, which uses every record)
    train_rows = torch.nonzero(replay["full"]).squeeze(1) if sp.cs is not None and n else None
    n_train = int(train_rows.numel()) if train_rows is not None else n
    # --eval-games: the net that played this iteration's self-play, to be matched against the trained one
    snapshot = copy.deepcopy(st.model) if getattr(args, "eval_games", 0) and rank == 0 else None
    losses = []
    if n_train and (not args.train_on_rank0 or rank == 0):
        g = torch.Generator(device="cuda").manual_seed(args.seed * 1000 + it)
        for k in range(args.train_steps):
            idx = torch.randint(0, n_train, (min(args.batch, n_train),), device="cuda", generator=g)
            if train_rows is not None:
                idx = train_rows[idx]
            planes, pi, z = train.make_batch(replay, idx, size=args.size, augment_seed=args.seed + 31 * it + k)
            losses.append(train.train_step(st.master, st.opt, planes, pi, z)["loss"])
        st._publish()
    ev[3].record()
    nbytes = bzd.broadcast_weights(st.model, src=0)
    if hasattr(st.evaluator, "refresh"):
        st.evaluator.refresh()  # in place: graph replays of the next iteration read the new weights
    ev[4].record()
    torch.cuda.synchronize()
    sp.mcts.check_errors()
    stats = sp.stats()
    ms = {"selfplay": ev[0].elapsed_time(ev[1]), "replay_gather": ev[1].elapsed_time(ev[2]),
          "train": ev[2].elapsed_time(ev[3]), "weight_broadcast": ev[3].elapsed_time(ev[4])}
    line = {
        "iteration": it, "world": world, "games_per_gpu": args.games, "sims_per_move": args.sims, "plies": args.plies,
        "leaves_per_iteration": args.leaves, "wall_s": time.perf_counter() - t0, "ms": ms,
        "sims_per_sec_per_gpu": args.games * args.sims * args.plies / (ms["selfplay"] * 1e-3),
        "replay_records_gathered": int(n), "local_records": int(shard["me"].shape[0]),
        "games_finished_local": stats["games"], "records_dropped_local": stats["dropped"],
        "train_steps": len(losses), "train_batch": min(args.batch, n_train) if n_train else 0,
        "loss_first_last": [losses[0], losses[-1]] if losses else None,
        "broadcast_bytes": nbytes, "replay_gather": gather_info,
    }
    if world > 1 and gather_info:
        # NCCL-tests convention: all-gather algbw = bytes every rank ends up with / time, busbw = algbw * (W-1)/W;
        # broadcast busbw = algbw.  The gather time also holds the shard packing and the (game, ply) sort.
        sec = ms["replay_gather"] * 1e-3
        line["replay_gather"]["algbw_GBps"] = gather_info["gathered_bytes"] / sec / 1e9
        line["replay_gather"]["busbw_GBps"] = gather_info["gathered_bytes"] * (world - 1) / world / sec / 1e9
        line["weight_broadcast_busbw_GBps"] = nbytes / (ms["weight_broadcast"] * 1e-3) / 1e9
    if sp.eg is not None:
        line["endgame"] = {"solve": sp.endgame_solve, "empties": sp.endgame_empties, "every": sp.endgame_every,
                           "games": stats["endgame_games"] - eg_stats0["endgame_games"],
                           "plies": stats["endgame_plies"] - eg_stats0["endgame_plies"],
                           "pending": stats["endgame_pending"],
                           "overflow": stats["endgame_overflow"] - eg_stats0["endgame_overflow"],
                           "ms": sp.endgame_ms() - eg_ms0}
    if resign_line is not None:
        resign_line["resigned_local"] = stats["resigned"] - rs_stats0["resigned"]
        resign_line["audited_local"] = stats["audited"] - rs_stats0["audited"]
        line["resign"] = resign_line
    if sp.cs is not None:
        line["cap"] = {"full_fraction": sp.full_fraction, "fast_sims": sp.fast_sims,
                       "full_plies_local": stats["full_plies"] - cap_stats0["full_plies"],
                       "fast_plies_local": stats["fast_plies"] - cap_stats0["fast_plies"],
                       "records_trained_on": n_train, "games_finished_local": stats["games"] - cap_stats0["games"]}
    if snapshot is not None:
        t_eval = time.perf_counter()
        r = match.BatchedMatch(st.model, snapshot, args.eval_games, args.sims, n_leaves=args.leaves, board_size=args.size,
                               seed=args.seed * 1000 + it).play()
        line["eval"] = {"score": r["score"], "elo": r["elo"], "elo_ci": r["elo_ci"], "wins": r["wins"], "draws": r["draws"],
                        "losses": r["losses"], "ms": (time.perf_counter() - t_eval) * 1e3}
        del snapshot
    if getattr(args, "eval_minimax", None) is not None and rank == 0:
        t_eval = time.perf_counter()
        r = match.BatchedMatch(st.model, match.Minimax(args.eval_minimax), args.eval_games, args.sims, n_leaves=args.leaves,
                               board_size=args.size, seed=args.seed * 1000 + it).play()
        line["eval_minimax"] = {"depth": int(args.eval_minimax), "score": r["score"], "elo": r["elo"], "elo_ci": r["elo_ci"],
                                "wins": r["wins"], "draws": r["draws"], "losses": r["losses"],
                                "minimax_nodes": r["minimax_nodes"], "ms": (time.perf_counter() - t_eval) * 1e3}
    if st.endgame_suite is not None:
        t_eval = time.perf_counter()
        r = endgame.evaluate(st.model, st.endgame_suite, (0, args.sims), args.leaves)
        line["eval_endgame"] = {"solve": "wld" if st.endgame_suite.wld else "exact", "empties": r["empties"],
                                "positions": r["positions"], "budgets": r["budgets"],
                                "random": r["baselines"]["random"], "ms": (time.perf_counter() - t_eval) * 1e3}
    if caught:
        line["warnings"] = [str(w.message) for w in caught]
    if args.checkpoint and rank == 0:
        path = checkpoint_path(args.checkpoint, it)
        extra = {"games_per_gpu": args.games, "sims_per_move": args.sims, "world": world}
        if sp.rs is not None:
            extra["resign_threshold"] = sp.resign_threshold
        if sp.cs is not None:
            extra["fast_sims"], extra["full_fraction"] = sp.fast_sims, sp.full_fraction
        train.save_checkpoint(path, st.master, st.opt, iteration=it + 1, extra=extra)
        line["checkpoint"] = path
    return line


def run(args) -> list[dict]:
    rank, world, local = bzd.init()
    if not torch.cuda.is_available():
        raise SystemExit("betazero_b200.loop needs CUDA devices: there is no CPU fallback")
    torch.cuda.set_device(local)
    st = LoopState(args, rank, world)
    out = []
    for it in range(st.first_iteration, st.first_iteration + args.iterations):
        line = run_iteration(st, it)
        out.append(line)
        if rank == 0:
            print(json.dumps(line), flush=True)
    return out


def main():
    d = default_args()
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=d.games)
    ap.add_argument("--sims", type=int, default=d.sims)
    ap.add_argument("--leaves", type=int, default=d.leaves, help="virtual-loss descents per tree and iteration (1 = sequential search)")
    ap.add_argument("--plies", type=int, default=d.plies, help="lockstep plies per iteration (a game lasts ~60)")
    ap.add_argument("--size", type=int, default=d.size)
    ap.add_argument("--iterations", type=int, default=d.iterations)
    ap.add_argument("--train-steps", type=int, default=d.train_steps)
    ap.add_argument("--batch", type=int, default=d.batch)
    ap.add_argument("--lr", type=float, default=d.lr)  # SL/train.py:190
    ap.add_argument("--temp-plies", type=int, default=d.temp_plies)
    ap.add_argument("--net", default=d.net)
    ap.add_argument("--hidden", type=int, default=d.hidden)
    ap.add_argument("--seed", type=int, default=d.seed)
    ap.add_argument("--train-on-rank0", action="store_true")
    ap.add_argument("--reuse", action="store_true", help="keep the searched subtree from move to move (bz_mcts_reroot): --sims "
                                                         "NEW simulations per move on top of the kept ones")
    ap.add_argument("--eval-games", type=int, default=d.eval_games,
                    help="rank 0 plays this many games (even) between the trained net and the net before training after "
                         "every iteration, with --sims / --leaves, and reports them as \"eval\" (0 = off)")
    ap.add_argument("--eval-minimax", type=int, default=d.eval_minimax, metavar="DEPTH",
                    help="rank 0 also plays --eval-games games between the trained net and the reference's minimax player "
                         "of this depth (0 .. 8) after every iteration, and reports them as \"eval_minimax\"")
    ap.add_argument("--eval-endgame", type=int, default=d.eval_endgame, metavar="EMPTIES",
                    help="rank 0: score the trained net's moves on 4096 positions with EMPTIES empty squares (at most 20) "
                         "against the exact solver, at 0 simulations and at --sims, and report them as \"eval_endgame\"")
    ap.add_argument("--endgame-empties", type=int, default=d.endgame_empties, metavar="E",
                    help="hand every self-play game to the exact endgame solver once a searched move leaves at most E "
                         "empty squares (1 .. 20; 0 = off): perfect play and exact z labels for the end of every game")
    ap.add_argument("--endgame-every", type=int, default=d.endgame_every, metavar="K",
                    help="with --endgame-empties: run a solver phase on the queued games every K plies")
    ap.add_argument("--endgame-solve", choices=selfplay.ENDGAME_SOLVES, default=d.endgame_solve,
                    help="the solver of --endgame-empties and --eval-endgame: exact (the final margin) or wld (win / "
                         "draw / loss only: cheaper; handover pi uniform over the moves that keep the result)")
    ap.add_argument("--resign", type=float, default=d.resign, metavar="V",
                    help="a self-play game that is not audited resigns at its first searched ply whose q (W / N of the "
                         "most visited root edge, the mover's view) is below V (-1 .. 1; -1 = audit only; default off)")
    ap.add_argument("--resign-audit", type=float, default=d.resign_audit, metavar="F",
                    help="with --resign: the fraction of games that never resign and measure its false positives")
    ap.add_argument("--resign-fp", type=float, default=d.resign_fp, metavar="P",
                    help="set the threshold after every iteration from its audited games: the largest one whose "
                         "false-positive rate stays at most P (switches resignation on, from --resign or -1)")
    ap.add_argument("--fast-sims", type=int, default=d.fast_sims, metavar="N",
                    help="randomized search budgets: plies that are not full are searched with N simulations (a "
                         "multiple of --leaves, 2 * leaves .. --sims; default off); only full plies are trained on")
    ap.add_argument("--full-fraction", type=float, default=d.full_fraction, metavar="P",
                    help="with --fast-sims: the fraction of plies searched with --sims (a Philox draw per ply)")
    ap.add_argument("--checkpoint", default=None, help="write a state_dict checkpoint (master weights + Adam state) here "
                                                       "after every iteration (rank 0); SL/train.py:204-214.  A {iteration} "
                                                       "in the path is replaced by the iteration number, so every "
                                                       "iteration's checkpoint is kept")
    ap.add_argument("--resume", default=None, help="continue from a checkpoint written by --checkpoint")
    args = ap.parse_args()
    if args.checkpoint:
        os.makedirs(os.path.dirname(os.path.abspath(args.checkpoint)), exist_ok=True)
    run(args)
    if bzd.world_size() > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
