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
adds ``eval_endgame``; the suite is drawn and solved once per run.
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
from . import endgame, match, mcts, minimax, net, selfplay, train


def default_args(**over) -> SimpleNamespace:
    """the command line's defaults as a namespace (for callers that drive iterations from Python: bench.py, tests)"""
    a = SimpleNamespace(games=4096, sims=800, leaves=4, plies=70, size=8, iterations=1, train_steps=8, batch=4096, lr=1e-4,
                        temp_plies=8, net="mlp", hidden=256, seed=0, train_on_rank0=False, checkpoint=None, resume=None,
                        reuse=False, eval_games=0, eval_minimax=None, eval_endgame=None)
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
        self.endgame_suite = None  # --eval-endgame: drawn and solved once per run (rank 0)
        ee = getattr(args, "eval_endgame", None)
        if ee is not None:
            if not 1 <= int(ee) <= minimax.SOLVE_MAX_EMPTIES:
                raise ValueError(f"eval_endgame must be in 1 .. {minimax.SOLVE_MAX_EMPTIES} empty squares; got {ee}")
            if rank == 0:
                self.endgame_suite = endgame.solve_suite(endgame.positions(ENDGAME_POSITIONS, int(ee), args.size, args.seed))
        self.model = net.make_net(args.net, hidden=args.hidden, seed=args.seed)
        self.master = net.make_net(args.net, hidden=args.hidden, seed=args.seed, dtype=torch.float32)  # fp32 master weights
        self.opt = torch.optim.Adam(self.master.parameters(), lr=args.lr)  # the reference's optimiser family (SL/train.py:87)
        self.first_iteration = 0
        if args.resume:
            self.first_iteration = train.load_checkpoint(args.resume, self.master, self.opt)
            self._publish()
        self.evaluator = (mcts.FusedNetEvaluator(self.model) if hasattr(self.model, "forward_raw")
                          else mcts.NetEvaluator(self.model))
        self.sp = selfplay.BatchedSelfPlay(args.games, args.sims, self.evaluator, board_size=args.size,
                                           temp_plies=args.temp_plies, seed=args.seed, rank=rank, world=world,
                                           n_leaves=args.leaves, reuse=bool(getattr(args, "reuse", False)),
                                           graph_unroll=min(16, max(1, args.sims // args.leaves - 1)))
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
    # --eval-games: the net that played this iteration's self-play, to be matched against the trained one
    snapshot = copy.deepcopy(st.model) if getattr(args, "eval_games", 0) and rank == 0 else None
    losses = []
    if n and (not args.train_on_rank0 or rank == 0):
        g = torch.Generator(device="cuda").manual_seed(args.seed * 1000 + it)
        for k in range(args.train_steps):
            idx = torch.randint(0, n, (min(args.batch, n),), device="cuda", generator=g)
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
        "train_steps": len(losses), "train_batch": min(args.batch, int(n)) if n else 0,
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
        line["eval_endgame"] = {"empties": r["empties"], "positions": r["positions"], "budgets": r["budgets"],
                                "random": r["baselines"]["random"], "ms": (time.perf_counter() - t_eval) * 1e3}
    if caught:
        line["warnings"] = [str(w.message) for w in caught]
    if args.checkpoint and rank == 0:
        path = checkpoint_path(args.checkpoint, it)
        train.save_checkpoint(path, st.master, st.opt, iteration=it + 1,
                              extra={"games_per_gpu": args.games, "sims_per_move": args.sims, "world": world})
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
