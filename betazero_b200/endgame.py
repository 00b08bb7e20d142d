"""Endgame accuracy: how often a net plays a perfect move, against the exact solver (``minimax.solve``).

A suite is a fixed, seeded set of positions with exactly ``empties`` empty squares (``positions``).  The solver gives
every legal move's exact final disc difference once; ``evaluate`` then scores the moves a net plays with its raw policy
(0 simulations: the first maximum of the legal logits, ``players.GreedyNetPlayer``'s rule) and with the one-launch
search (the most visited move, lowest id on ties: the rule of matches), per budget:

    move_accuracy        the played move's value equals the best value
    wld_accuracy         the played move keeps the sign of the best value (win / draw / loss)
    mean_disc_loss       best value minus the played move's value
    value_sign_accuracy  (budget 0) the value head's sign equals the exact outcome's, over decided positions
    value_mse            (budget 0) the value head against the exact outcome in {-1, 0, 1}

next to the random player's expected scores (exact, from the move values) and ``Minimax(d)``'s moves
(``minimax.best_moves``).  No opponent and no game noise: with a fixed seed a number means the same in every run.

A win/draw/loss suite (``Suite.wld``, ``--wld``) is solved by ``minimax.solve(wld=True)``: its move values are only
signs, so every move score is ``wld_accuracy`` alone (``move_accuracy`` and ``mean_disc_loss`` are absent); the value
metrics use only signs and are those of the exact suite.

    python -m betazero_b200.endgame A.pt B.pt --empties 12 --positions 4096 --sims 0,800 --minimax 2,4
"""
from __future__ import annotations

import argparse
import json
from dataclasses import dataclass

import numpy as np
import torch

from . import env, mcts, minimax

GAMES_PER_BATCH = 4096  # random games played side by side while a suite is drawn


@dataclass
class Suite:
    """mover-relative positions (int64 CUDA tensors of uint64 bitboards) and, once ``solve_suite`` ran, the solver's
    results: value int8 [n], move_value int8 [n, 65], nodes int64 [n] (numpy), and the solve's time.  ``wld``: solve
    for win / draw / loss only (the values are signs)"""
    me: torch.Tensor
    opp: torch.Tensor
    size: int
    empties: int
    seed: int
    wld: bool = False
    value: np.ndarray | None = None
    move_value: np.ndarray | None = None
    nodes: np.ndarray | None = None
    solve_ms: float | None = None

    def __len__(self) -> int:
        return self.me.numel()


def _popcount(x: np.ndarray) -> np.ndarray:
    return np.unpackbits(np.ascontiguousarray(x, np.uint64).view(np.uint8).reshape(-1, 8), axis=1).sum(1)


def positions(n: int, empties: int, size: int = 8, seed: int = 0, device="cuda") -> Suite:
    """``n`` positions with exactly ``empties`` empty squares whose mover has at least 2 legal moves (a forced move says
    nothing about accuracy).  Random games from the start position, choices drawn by ``numpy.random.default_rng(seed)``
    and rules from the env kernels; from each game the first position with ``empties`` empties and a mover who has a
    move is kept if that mover has 2 or more.  Games are played ``GAMES_PER_BATCH`` at a time until ``n`` positions are
    kept, in game order: the same seed gives the same suite."""
    if size not in (4, 6, 8):
        raise ValueError("size must be 4, 6 or 8 (Reversi)")
    if not 1 <= empties <= size * size - 5:
        raise ValueError(f"empties must be in 1 .. {size * size - 5} on {size}x{size}")
    rng = np.random.default_rng(seed)
    kept_me, kept_opp = [], []
    have = 0
    while have < n:
        B = GAMES_PER_BATCH
        me, opp, _ = env.reversi_init(B, size, device)
        active = np.ones(B, bool)
        found_me, found_opp = np.zeros(B, np.uint64), np.zeros(B, np.uint64)
        found = np.zeros(B, bool)
        while active.any():
            mask = env.to_host_u64(env.legal_mask(me, opp, size))
            mask_opp = env.to_host_u64(env.legal_mask(opp, me, size))
            h_me, h_opp = env.to_host_u64(me), env.to_host_u64(opp)
            e = size * size - _popcount(h_me | h_opp)
            moves = _popcount(mask)
            u = rng.random(B)  # one draw per game and ply, used or not: the stream does not depend on outcomes
            over = (moves == 0) & (mask_opp == 0)
            at = active & (e == empties) & (moves > 0)
            keep = at & (moves >= 2)
            found_me[keep], found_opp[keep], found[keep] = h_me[keep], h_opp[keep], True
            active &= ~(at | over | (e < empties))
            k = np.minimum((u * moves).astype(np.int64), np.maximum(moves - 1, 0))
            action = np.full(B, 64, np.uint8)  # a pass when there is no move
            for i in np.nonzero(active & (moves > 0))[0]:
                m = int(mask[i])
                for _ in range(int(k[i])):
                    m &= m - 1
                action[i] = (m & -m).bit_length() - 1
            me, opp, _ = env.apply(me, opp, torch.from_numpy(action).to(device), size)
        idx = np.nonzero(found)[0][: n - have]
        kept_me.append(found_me[idx])
        kept_opp.append(found_opp[idx])
        have += idx.size
    return Suite(env.to_device_u64(np.concatenate(kept_me), device), env.to_device_u64(np.concatenate(kept_opp), device),
                 size, empties, seed)


def solve_suite(suite: Suite) -> Suite:
    """fills the suite's exact (or, ``suite.wld``, win/draw/loss) values (once; a solved suite is returned as it is)"""
    if suite.move_value is not None:
        return suite
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    _, v, mv, nodes = minimax.solve(suite.me, suite.opp, suite.size, wld=suite.wld)
    e1.record()
    torch.cuda.synchronize()
    suite.solve_ms = e0.elapsed_time(e1)
    suite.value, suite.move_value, suite.nodes = v.cpu().numpy(), mv.cpu().numpy(), nodes.cpu().numpy()
    return suite


def move_metrics(move_value: np.ndarray, value: np.ndarray, played: np.ndarray, wld: bool = False) -> dict:
    """accuracy of the played moves (cell ids) against the exact move values (``wld``: against their signs, so only
    ``wld_accuracy``)"""
    mv = move_value.astype(np.int64)
    best = value.astype(np.int64)
    pv = mv[np.arange(len(played)), np.asarray(played, np.int64)]
    if (pv == -128).any():
        raise ValueError("a played move is not legal")
    out = {"wld_accuracy": float(np.mean(np.sign(pv) == np.sign(best)))}
    if not wld:
        out = {"move_accuracy": float(np.mean(pv == best)), **out, "mean_disc_loss": float(np.mean(best - pv))}
    return out


def random_metrics(move_value: np.ndarray, value: np.ndarray, wld: bool = False) -> dict:
    """the random player's expected scores: every legal move equally likely (``wld``: ``wld_accuracy`` only)"""
    mv = move_value.astype(np.int64)
    best = value.astype(np.int64)[:, None]
    legal = mv != -128
    n_legal = legal.sum(1)
    out = {"wld_accuracy": float(np.mean(((np.sign(mv) == np.sign(best)) & legal).sum(1) / n_legal))}
    if not wld:
        out = {"move_accuracy": float(np.mean(((mv == best) & legal).sum(1) / n_legal)), **out,
               "mean_disc_loss": float(np.mean(np.where(legal, best - mv, 0).sum(1) / n_legal))}
    return out


def value_metrics(head: np.ndarray, value: np.ndarray) -> dict:
    """the value head (tanh, the mover's view) against the exact outcome"""
    z = np.sign(value.astype(np.int64))
    decided = z != 0
    return {"value_sign_accuracy": float(np.mean(np.sign(head[decided]) == z[decided])) if decided.any() else None,
            "value_mse": float(np.mean((head.astype(np.float64) - z) ** 2))}


@torch.no_grad()
def raw_policy(net, me: torch.Tensor, opp: torch.Tensor, size: int = 8):
    """(moves int64 [n], value head float64 [n]): the first maximum of the legal logits, GreedyNetPlayer's rule"""
    mask = env.to_host_u64(env.legal_mask(me, opp, size))
    logits, v = net(env.planes(me, opp))
    logits = logits[:, :64].float().cpu().numpy()
    legal = ((mask[:, None] >> np.arange(64, dtype=np.uint64)) & np.uint64(1)).astype(bool)
    return np.argmax(np.where(legal, logits, -np.inf), axis=1), v.double().cpu().numpy()


def searched_moves(net, me: torch.Tensor, opp: torch.Tensor, sims: int, n_leaves: int = 4, size: int = 8) -> np.ndarray:
    """the one-launch search's most visited move of every position (lowest id on ties), as a match plays it"""
    pools = mcts.TreePools(me.numel(), sims, game=mcts.GAME_REVERSI, board_size=size, n_leaves=n_leaves)
    search = mcts.BatchedMCTS(pools, mcts.FusedNetEvaluator(net), use_graph=False)
    search.search(me, opp, sims)
    return search.best_action().long().cpu().numpy()


def evaluate(net, suite: Suite, sims=(0, 800), n_leaves: int = 4, minimax_depths=()) -> dict:
    """the net's endgame accuracy on the suite, per simulation budget, with the baselines (the suite is solved first if
    it is not yet)"""
    solve_suite(suite)
    out = {"positions": len(suite), "empties": suite.empties, "size": suite.size, "seed": suite.seed, "budgets": {}}
    for s in sims:
        s = int(s)
        if s == 0:
            played, head = raw_policy(net, suite.me, suite.opp, suite.size)
            r = move_metrics(suite.move_value, suite.value, played, suite.wld)
            r.update(value_metrics(head, suite.value))
        else:
            r = move_metrics(suite.move_value, suite.value, searched_moves(net, suite.me, suite.opp, s, n_leaves, suite.size),
                             suite.wld)
        out["budgets"][str(s)] = r
    out["baselines"] = baselines(suite, minimax_depths)
    return out


def baselines(suite: Suite, minimax_depths=()) -> dict:
    solve_suite(suite)
    out = {"random": random_metrics(suite.move_value, suite.value, suite.wld)}
    keys = torch.arange(len(suite), dtype=torch.int64, device=suite.me.device)
    for d in minimax_depths:
        a, _, _ = minimax.best_moves(suite.me, suite.opp, int(d), suite.size, seed=suite.seed, keys=keys)
        out[f"minimax{int(d)}"] = move_metrics(suite.move_value, suite.value, a.long().cpu().numpy(), suite.wld)
    return out


def solve_stats(suite: Suite) -> dict:
    solve_suite(suite)
    return {"solve": "wld" if suite.wld else "exact", "ms": suite.solve_ms, "nodes": int(suite.nodes.sum()),
            "max_nodes": int(suite.nodes.max())}


def main(argv=None):
    ap = argparse.ArgumentParser(prog="python -m betazero_b200.endgame", description=__doc__.split("\n\n")[0])
    ap.add_argument("checkpoints", nargs="*", help="state_dict checkpoints (betazero_b200.train.save_checkpoint)")
    ap.add_argument("--empties", type=int, default=12)
    ap.add_argument("--positions", type=int, default=4096)
    ap.add_argument("--sims", default="0,800", help="simulation budgets, comma-separated (0 = the raw policy)")
    ap.add_argument("--minimax", default="", help="Minimax depths for baselines, comma-separated")
    ap.add_argument("--size", type=int, default=8)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--leaves", type=int, default=4, help="virtual-loss descents per tree and iteration of the search")
    ap.add_argument("--wld", action="store_true", help="solve for win / draw / loss only (cheaper; the move scores are "
                                                       "wld_accuracy alone)")
    args = ap.parse_args(argv)
    from . import train

    sims = [int(x) for x in args.sims.split(",") if x.strip()]
    depths = [minimax.check_depth(x) for x in args.minimax.split(",") if x.strip()]
    if args.empties > minimax.SOLVE_MAX_EMPTIES:
        raise SystemExit(f"--empties must be at most {minimax.SOLVE_MAX_EMPTIES}")
    suite = positions(args.positions, args.empties, args.size, args.seed)
    suite.wld = args.wld
    solve_suite(suite)
    out = {"size": args.size, "empties": args.empties, "positions": len(suite), "seed": args.seed, "leaves": args.leaves,
           "solve": solve_stats(suite), "baselines": baselines(suite, depths), "checkpoints": {}}
    for path in args.checkpoints:
        r = evaluate(train.load_net(path), suite, sims, args.leaves)
        out["checkpoints"][path] = r["budgets"]
    print(json.dumps(out), flush=True)
    return out


if __name__ == "__main__":
    main()
