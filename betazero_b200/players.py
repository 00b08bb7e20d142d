"""Drop-in players: ``get_move(board) -> (row, col)`` backed by the batched GPU MCTS.

The reference defines the search interface as an ABC with one method
(``ReversiPlayer.get_move`` src/reversi/players/reversi_players.py:5-8, ``Player.get_move``
src/tic_tac_toe/players.py:6-9) and ships random / minimax / policy-net players behind it, but no
MCTS.  ``MCTSPlayer`` / ``TicTacToeMCTSPlayer`` fill that hole and plug into the reference's game
managers unchanged (``ReversiTerminal(p1, p2).play()`` reversi_terminal.py:10-38,
``TicTacToeHeadless(p1, p2).play()`` tic_tac_toe.py:6-34).  Conventions kept from the reference:
Reversi players hold ``self.symbol`` in {+1, -1} (reversi_players.py:27-28) and return
``(None, None)`` when there is no move (:32); the move is the most visited action with the lowest
row-major index on ties (the argmax-over-legal pick of players.py:92-98).

A single ``get_move`` searches ONE tree -- that is the compatibility boundary, not the fast path;
throughput comes from ``betazero_b200.selfplay.BatchedSelfPlay`` (thousands of trees per launch).
"""
from __future__ import annotations

from abc import ABC, abstractmethod

import numpy as np
import torch

from . import env, mcts, minimax
from .boards import _grid_to_bits


class ReversiPlayer(ABC):
    """reversi_players.py:5-8"""

    @abstractmethod
    def get_move(self, board):
        pass


class Player(ABC):
    """src/tic_tac_toe/players.py:6-9"""

    @abstractmethod
    def get_move(self, board):
        pass


def _make_evaluator(evaluator, net, salt):
    if evaluator is not None:
        return evaluator
    if net is not None:
        return mcts.FusedNetEvaluator(net) if hasattr(net, "forward_raw") else mcts.NetEvaluator(net)
    return mcts.HashEvaluator(salt)


class MCTSPlayer(ReversiPlayer):
    """AlphaZero-style MCTS player for Reversi (sizes 4, 6, 8).

    ``net``: a policy/value module from ``betazero_b200.net`` (or pass ``evaluator``); with neither,
    the deterministic hash pseudo-net is used (parity / tests)."""

    def __init__(self, symbol, net=None, n_sims: int = 100, c_puct: float = 1.25, size: int = 8, evaluator=None,
                 salt: int = 0, n_leaves: int = 1, reuse: bool = False):
        self.symbol = symbol  # 1 for X, -1 for O
        self.n_sims, self.size = int(n_sims), int(size)
        # n_leaves > 1: virtual-loss descents per iteration (n_sims must be a multiple); 1 = the sequential search
        # reuse: keep the subtree of (own move, opponent's reply) from one get_move to the next (oracle/mcts_ref.py
        # MCTS.advance); every call then adds n_sims simulations to what the previous searches left below the new root
        self.reuse = bool(reuse)
        self.pools = mcts.TreePools(1, self.n_sims, game=mcts.GAME_REVERSI, board_size=size, c_puct=c_puct, n_leaves=n_leaves,
                                    reuse=self.reuse)
        self.search = mcts.BatchedMCTS(self.pools, _make_evaluator(evaluator, net, salt), use_graph=False)
        self.last_counts = None
        self.last_policy = None
        self.last_inherited = 0   # visits the root of the last search started with (reuse)
        self._after_own = None    # (me, opp) device tensors + occupancy after this player's last move, opponent to move
        self._own_action = None

    def _continue_or_reset(self, me_t, opp_t, me: int, opp: int) -> None:
        """reuse: follow the own move and the opponent's reply (a new disc, or a pass) down the kept tree"""
        if self._after_own is not None:
            pm, po_, occ = self._after_own
            new = (me | opp) & ~occ
            if new == 0 or (new & (new - 1)) == 0:  # one reply (or a pass); anything else: not the same game, start over
                b = 64 if new == 0 else new.bit_length() - 1
                self.search.advance(self._own_action, pm, po_)
                self.search.advance(torch.tensor([b], dtype=torch.uint8, device=me_t.device), me_t, opp_t)
                return
        self.search.reset(me_t, opp_t)

    def get_move(self, board):
        if int(board.size) != self.size:
            raise ValueError(f"this player was built for {self.size}x{self.size} boards")
        me, opp = _grid_to_bits(np.asarray(board.board), self.symbol, 8)
        me_t, opp_t = env.to_device_u64(np.array([me], np.uint64)), env.to_device_u64(np.array([opp], np.uint64))
        if self.reuse:
            self._continue_or_reset(me_t, opp_t, me, opp)
            self.last_inherited = int(self.pools.inherited[0].item())
            self.search.run(self.n_sims)
            cnt, pi, _ = self.search.root_policy()
            self.search.check_errors()
        else:
            cnt, pi, _ = self.search.search(me_t, opp_t, self.n_sims)
        best = self.search.best_action()
        a = int(best[0].item())
        self.last_counts = cnt[0].cpu().numpy().copy()
        self.last_policy = pi[0].cpu().numpy().copy()
        if self.reuse:
            if a <= 64:
                pm, po_, _ = env.apply(me_t, opp_t, best.clone(), self.size)
                occ = (me | opp) | ((1 << a) if a < 64 else 0)
                self._after_own, self._own_action = (pm, po_, occ), best.clone()
            else:
                self._after_own = None
        if a >= 64:  # pass (64) or finished game (255): the reference convention for "no moves"
            return None, None
        return a >> 3, a & 7


class TicTacToeMCTSPlayer(Player):
    """MCTS player for the reference's tic-tac-toe loop (BASELINE config 1)."""

    def __init__(self, symbol, net=None, n_sims: int = 100, c_puct: float = 1.25, evaluator=None, salt: int = 0,
                 n_leaves: int = 1):
        self.symbol = symbol
        self.n_sims = int(n_sims)
        self.pools = mcts.TreePools(1, self.n_sims, game=mcts.GAME_TTT, c_puct=c_puct, n_leaves=n_leaves)
        self.search = mcts.BatchedMCTS(self.pools, _make_evaluator(evaluator, net, salt), use_graph=False)
        self.last_counts = None
        self.last_policy = None

    def get_move(self, board):
        me, opp = _grid_to_bits(np.asarray(board.board), self.symbol, 3)
        cnt, pi, _ = self.search.search(env.to_device_u64(np.array([me], np.uint64)),
                                        env.to_device_u64(np.array([opp], np.uint64)), self.n_sims)
        a = int(self.search.best_action()[0].item())
        self.last_counts = cnt[0].cpu().numpy().copy()
        self.last_policy = pi[0].cpu().numpy().copy()
        if a >= 9:
            return None, None
        return a // 3, a % 3


class GreedyNetPlayer(ReversiPlayer):
    """The reference's AIPlayer.get_move (players.py:84-98) for Reversi: canonicalise with
    ``symbol * board`` (:85), run the net once, take the best LEGAL move (first maximum in
    row-major order).  Input goes through the K6 plane kernel, legality through K1."""

    def __init__(self, symbol, net, size: int = 8):
        self.symbol, self.net, self.size = symbol, net, int(size)

    @torch.no_grad()
    def get_move(self, board):
        me_i, opp_i = _grid_to_bits(np.asarray(board.board), self.symbol, 8)
        me = env.to_device_u64(np.array([me_i], np.uint64))
        opp = env.to_device_u64(np.array([opp_i], np.uint64))
        mask = int(env.to_host_u64(env.legal_mask(me, opp, self.size))[0])
        if mask == 0:
            return None, None
        logits, _ = self.net(env.planes(me, opp))
        logits = logits[0, :64].float().cpu().numpy()
        legal = np.array([(mask >> a) & 1 for a in range(64)], dtype=bool)
        a = int(np.argmax(np.where(legal, logits, -np.inf)))
        return a >> 3, a & 7


class AIPlayer(ReversiPlayer):
    """The reference's ``AIPlayer(path_to_model, symbol)`` (src/tic_tac_toe/players.py:77-98) for this engine's
    checkpoints: built from a model FILE, plays the net's best legal move (:92-98).  The file is a state_dict
    checkpoint written by ``betazero_b200.train.save_checkpoint`` (the reference pickles the whole module, :80 /
    SL/train.py:214, which needs the defining source on the import path and arbitrary-code unpickling).
    ``n_sims > 0`` puts the batched MCTS in front of the same net (what the AlphaZero loop's arena wants)."""

    def __init__(self, path_to_model, symbol, n_sims: int = 0, size: int = 8, c_puct: float = 1.25, n_leaves: int = 1,
                 device="cuda"):
        from . import train

        self.model = train.load_net(path_to_model, device=device)
        self.symbol, self.size = symbol, int(size)
        if n_sims > 0:
            self._impl = MCTSPlayer(symbol, net=self.model, n_sims=n_sims, c_puct=c_puct, size=size, n_leaves=n_leaves)
        else:
            self._impl = GreedyNetPlayer(symbol, self.model, size=size)

    def get_move(self, board):
        return self._impl.get_move(board)


class OptimalPlayer(ReversiPlayer):
    """The reference's depth-limited minimax ``OptimalPlayer(symbol, max_depth)`` (reversi_players.py:35-77) on the GPU
    kernel (``bz_minimax_moves``): disc-difference evaluation, first best move in row-major order, no pass handling
    inside the search.  Where the search returns no move (``max_depth = 0``, or every move worth -inf) the reference
    plays ``random.choice`` (:42-43); here that move is drawn with Philox keyed by ``seed`` and ``game_key`` and counted
    by the discs on the board, so a game replays exactly (oracle/minimax_ref.py).  ``(None, None)`` when there is no
    move (:32)."""

    def __init__(self, symbol, max_depth: int, size: int = 8, seed: int = 0, game_key: int = 0):
        self.symbol, self.max_depth = symbol, minimax.check_depth(max_depth)
        self.size, self.seed, self.game_key = int(size), int(seed), int(game_key)
        self.last_value = None
        self.last_nodes = None

    def get_move(self, board):
        if int(board.size) != self.size:
            raise ValueError(f"this player was built for {self.size}x{self.size} boards")
        me, opp = _grid_to_bits(np.asarray(board.board), self.symbol, 8)
        a, v, n = minimax.best_moves(env.to_device_u64(np.array([me], np.uint64)),
                                     env.to_device_u64(np.array([opp], np.uint64)), self.max_depth, self.size, self.seed,
                                     self.game_key)
        a = int(a[0].item())
        self.last_value, self.last_nodes = int(v[0].item()), int(n[0].item())
        if a >= 64:  # pass (64) or finished game (255)
            return None, None
        return a >> 3, a & 7


class RandomPlayer(OptimalPlayer):
    """The reference's ``RandomPlayer(symbol)`` (reversi_players.py:26-32): a uniformly random legal move, here the
    Philox move of ``OptimalPlayer`` at depth 0."""

    def __init__(self, symbol, size: int = 8, seed: int = 0, game_key: int = 0):
        super().__init__(symbol, 0, size=size, seed=seed, game_key=game_key)


class PerfectPlayer(ReversiPlayer):
    """The perfect player of the endgame: the exact solver's move (``minimax.solve``, ``bz_endgame_solve``), the first
    move in row-major order that reaches the best final disc difference.  It takes boards with at most 20 empty squares
    (``ValueError`` otherwise) and returns ``(None, None)`` when there is no move (reversi_players.py:32)."""

    def __init__(self, symbol, size: int = 8):
        self.symbol, self.size = symbol, int(size)
        self.last_value = None
        self.last_nodes = None

    def get_move(self, board):
        if int(board.size) != self.size:
            raise ValueError(f"this player was built for {self.size}x{self.size} boards")
        me, opp = _grid_to_bits(np.asarray(board.board), self.symbol, 8)
        a, v, _, n = minimax.solve(env.to_device_u64(np.array([me], np.uint64)),
                                   env.to_device_u64(np.array([opp], np.uint64)), self.size)
        a = int(a[0].item())
        self.last_value, self.last_nodes = int(v[0].item()), int(n[0].item())
        if a >= 64:  # pass (64) or finished game (255)
            return None, None
        return a >> 3, a & 7
