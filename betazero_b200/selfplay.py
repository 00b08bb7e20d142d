"""Batched lockstep self-play: the reference episode loop (reversi_terminal.py:16-38) for
thousands of concurrent games per GPU.

Per ply, for ALL game slots at once:
    search (BatchedMCTS: n_sims iterations) -> bz_selfplay_advance (pick move from root visit
    counts, record (board, pi), apply / pass, terminal test, score + flush finished games to the
    replay buffer, restart the slot) -> next search from the new positions.
Games shard embarrassingly: rank r of W owns game ids {r*B + s + k*W*B}; move sampling is keyed by
(seed, game id, ply), so a game's content does not depend on which GPU / slot played it.

Endgame handover (opt-in, ``endgame_empties=E``): a game whose searched move leaves at most E empty squares moves to a
device-side queue and its slot restarts; every ``endgame_every`` plies the exact solver plays every queued game to its end
(bz_selfplay_advance_endgame, bz_selfplay_endgame_play).  Its records up to the handover are those the game has without
the feature, the solver's records carry pi uniform over the optimal moves, and every z is the exact outcome of the
handover position.  ``endgame_solve="wld"`` hands the games to the win/draw/loss solver instead (bz_selfplay_endgame_play_wld):
cheaper, with the same z, but pi is uniform over every move that keeps the result rather than over the moves that
maximise the final margin -- a label with less information, which is why the exact solver stays the default.

Resignation (opt-in, ``resign_threshold=v``): a game that is not audited resigns at its first searched ply whose q -- W / N
of the most visited root edge, the mover's view -- is below v; the ply is recorded, the mover loses and the slot
restarts (bz_selfplay_advance_resign).  A fraction ``resign_audit`` of the games (by a Philox draw on the game id) never
resigns: they measure how often resigning would have been wrong (``resign.false_positive_rate``, ``resign.calibrate``).
Every record then carries its ply's q (NaN for solver-played plies) and ``drain_replay`` returns it as "q".  The
threshold can change between plies (``set_resign_threshold``): the state is passed by value at every launch.

Randomized search budgets (opt-in, ``fast_sims=n``; KataGo's playout cap randomization): a ply of game g at ply t is full
iff a Philox draw on (seed, g, 0x80000000 | t) falls below ``full_fraction``; a full ply is searched with ``n_sims``, any
other ply with ``fast_sims``, both from a fresh tree.  Every record carries ``full`` (solver-played records are full) and
``drain_replay`` returns it as "full": the policy target of a fast ply comes from a cheap search and is not trained on,
its z is the game's.  Each ply runs bz_selfplay_cap_layout (the full slots' trees first, padded to a CTA pair, then the
fast ones), bz_mcts_reset from its roots, bz_mcts_search_fused_entrants with the two budgets, and
bz_selfplay_advance_cap; launches made of fast pairs only end early.  Root noise, when on, perturbs full plies only.
It needs the one-launch search and refuses tree reuse.
"""
from __future__ import annotations

import ctypes as C

import math

import torch

from . import _lib
from . import resign as _resign
from ._lib import BzSelfplayCapState, BzSelfplayEndgameState, BzSelfplayResignState, BzSelfplayState
from .mcts import BatchedMCTS, FusedNetEvaluator, TreePools

N_ACTIONS = 65
SOLVE_MAX_EMPTIES = 20  # BZ_SOLVE_MAX_EMPTIES
ENDGAME_SOLVES = ("exact", "wld")
PAIR_TREES = 56  # BZ_MATCH_TREES_PER_PAIR: the trees of a CTA pair of the one-launch search
FULL_COUNTER = 0x80000000  # the Philox counter of the full-ply draw is 0x80000000 | ply


def full_below(fraction) -> int:
    """floor(fraction * 2^32) for a full fraction in [0, 1]"""
    f = float(fraction)
    if not 0.0 <= f <= 1.0:
        raise ValueError(f"full_fraction must be in [0, 1]; got {fraction}")
    return int(math.floor(f * 2.0 ** 32))


def check_fast_sims(fast_sims, n_sims: int, n_leaves: int) -> int:
    """2 K <= fast_sims <= n_sims, a multiple of K = n_leaves"""
    f, k = int(fast_sims), int(n_leaves)
    if not 2 * k <= f <= int(n_sims) or f % k:
        raise ValueError(f"fast_sims must be a multiple of n_leaves = {k} in {2 * k} .. n_sims = {n_sims}; got {fast_sims}")
    return f


def is_full(game_id: torch.Tensor, ply: torch.Tensor, seed: int, fraction: float) -> torch.Tensor:
    """bool tensor: the searches of these (game id, ply) plies are full (bz_philox_u32 on the device)"""
    L = _lib.load()
    g = game_id.to(device="cuda", dtype=torch.int64).contiguous()
    t = (ply.to(device="cuda", dtype=torch.int64) - FULL_COUNTER).to(torch.int32).contiguous()  # int32 bits of 0x80000000 | ply
    out = torch.empty(g.numel(), dtype=torch.int32, device="cuda")
    _lib.check(L.bz_philox_u32(int(seed), _lib.dptr(g), _lib.dptr(t), _lib.dptr(out), g.numel(), _lib.stream_ptr()),
               "bz_philox_u32")
    return (out.to(torch.int64) & 0xFFFFFFFF) < full_below(fraction)


def check_endgame_empties(empties, board_size: int) -> int:
    """0 (off) or 1 .. min(20, size^2 - 5): the start position is always searched"""
    e, hi = int(empties), min(SOLVE_MAX_EMPTIES, int(board_size) ** 2 - 5)
    if e != 0 and not 1 <= e <= hi:
        raise ValueError(f"endgame_empties must be 0 (off) or in 1 .. {hi} on a {board_size}x{board_size} board; got {empties}")
    return e


def check_endgame_solve(solve) -> str:
    """"exact" (bz_selfplay_endgame_play) or "wld" (bz_selfplay_endgame_play_wld)"""
    if solve not in ENDGAME_SOLVES:
        raise ValueError(f"endgame_solve must be one of {ENDGAME_SOLVES}; got {solve!r}")
    return solve


class BatchedSelfPlay:
    def __init__(self, n_games: int, n_sims: int, evaluator, board_size: int = 8, c_puct: float = 1.25,
                 temp_plies: int = 0, seed: int = 0, replay_cap: int | None = None, rank: int = 0, world: int = 1,
                 arena_units: int | None = None, use_graph: bool = True, graph_unroll: int = 16,
                 dirichlet_alpha: float = 0.0, dirichlet_eps: float = 0.25, n_leaves: int = 1, device="cuda",
                 one_launch: bool | None = None, reuse: bool = False, endgame_empties: int = 0, endgame_every: int = 8,
                 endgame_cap: int | None = None, endgame_solve: str = "exact", resign_threshold: float | None = None,
                 resign_audit: float = 0.1, fast_sims: int | None = None, full_fraction: float = 0.25):
        self.n_games, self.n_sims, self.board_size = int(n_games), int(n_sims), int(board_size)
        # randomized search budgets: checked before anything touches the GPU
        self.fast_sims, self.full_fraction = None, float(full_fraction)
        if fast_sims is not None:
            self._full_below = full_below(full_fraction)
            self.fast_sims = check_fast_sims(fast_sims, n_sims, n_leaves)
            if n_sims % int(n_leaves):
                raise ValueError(f"n_sims {n_sims} is not a multiple of n_leaves {n_leaves}")
            if reuse:
                raise ValueError("fast_sims does not combine with tree reuse: the layout gives a slot another tree from "
                                 "ply to ply, so there is no subtree to keep")
            if one_launch is False or int(n_leaves) not in (1, 2, 4) or not isinstance(evaluator, FusedNetEvaluator):
                raise ValueError("fast_sims needs the one-launch search (bz_mcts_search_fused_entrants): n_leaves 1, 2 "
                                 "or 4 and a FusedNetEvaluator on the bf16 MLP")
        self.resign_audit = float(resign_audit)
        self._audit_below = _resign.audit_below(resign_audit)
        if resign_threshold is not None:
            resign_threshold = _resign.check_threshold(resign_threshold)
        self.endgame_empties = check_endgame_empties(endgame_empties, board_size)
        self.endgame_solve = check_endgame_solve(endgame_solve)
        self.endgame_every = int(endgame_every)
        if self.endgame_every < 1:
            raise ValueError(f"endgame_every must be >= 1; got {endgame_every}")
        self.endgame_cap = int(endgame_cap if endgame_cap is not None else max(self.n_games, 1))
        if not 1 <= self.endgame_cap <= 1 << 22:
            raise ValueError(f"endgame_cap must be in 1 .. 2^22; got {endgame_cap}")
        self.rank, self.world = int(rank), int(world)
        self.device = torch.device(device)
        # reuse: a move's search continues on the subtree of the move played (opt-in; bz_mcts_reroot) -- n_sims MORE
        # simulations per move on top of the kept ones; the default is a fresh tree per move, which the goldens pin
        self.reuse = bool(reuse)
        self._moves = 0
        # randomized budgets: n_games + 55 trees, so the full range's padding to a CTA pair always fits
        n_trees = n_games + PAIR_TREES - 1 if self.fast_sims is not None else n_games
        self.pools = TreePools(n_trees, n_sims, board_size=board_size, c_puct=c_puct, arena_units=arena_units,
                               n_leaves=n_leaves, device=device, reuse=reuse)
        self.mcts = BatchedMCTS(self.pools, evaluator, use_graph=use_graph, graph_unroll=graph_unroll,
                                dirichlet_alpha=dirichlet_alpha, dirichlet_eps=dirichlet_eps,
                                noise_seed=seed * 7919 + rank, one_launch=one_launch)
        if self.fast_sims is not None and not self.mcts.one_launch_ok():
            raise ValueError("fast_sims needs the one-launch search (bz_mcts_search_fused_entrants): the evaluator's net "
                             "must run through the bf16 MLP kernel path")
        self.max_plies = 128
        B, H = max(self.n_games, 1), max(self.n_games, 1) * self.max_plies
        self.replay_cap = int(replay_cap if replay_cap is not None else B * 2 * self.max_plies)
        R = max(self.replay_cap, 1)
        dev = self.device

        def e(n, dt):
            return torch.empty(n, dtype=dt, device=dev)

        self.me, self.opp = e(B, torch.int64), e(B, torch.int64)
        self.player, self.ply, self.game_id = e(B, torch.int8), e(B, torch.int32), e(B, torch.int64)
        self.hist_me, self.hist_opp = e(H, torch.int64), e(H, torch.int64)
        self.hist_player, self.hist_action = e(H, torch.int8), e(H, torch.uint8)
        self.hist_pi = e(H * N_ACTIONS, torch.float32)
        self.rp_me, self.rp_opp = e(R, torch.int64), e(R, torch.int64)
        self.rp_pi = e(R * N_ACTIONS, torch.float32)
        self.rp_z, self.rp_game, self.rp_ply = e(R, torch.int8), e(R, torch.int64), e(R, torch.int16)
        self.counters = torch.zeros(8, dtype=torch.int64, device=dev)
        self.last_action = torch.zeros(B, dtype=torch.uint8, device=dev)
        s = BzSelfplayState()
        s.n_games, s.board_size, s.max_plies, s.temp_plies = self.n_games, self.board_size, self.max_plies, int(temp_plies)
        s.seed, s.id_stride, s.replay_cap = int(seed), self.world * self.n_games, self.replay_cap
        for name, _ in BzSelfplayState._fields_[7:]:
            setattr(s, name, getattr(self, name).data_ptr())
        self.c_struct = s
        self._ref = C.byref(s)
        self._L = _lib.load()
        self.launches = 0
        self._dropped_seen = 0  # counters[5] at the last drain (overflow is reported, never silent)
        _lib.check(self._L.bz_selfplay_init(self._ref, self.rank * self.n_games, _lib.stream_ptr()), "bz_selfplay_init")
        self.launches += 1
        self.eg = None
        self._advances = 0
        self._eg_events = []  # (start, end) CUDA events of the solver phases not yet summed
        self._eg_ms = 0.0
        if self.endgame_empties:
            self._init_endgame()
        self.rs = None
        if resign_threshold is not None:
            self._init_resign(resign_threshold)
        self.cs = None
        if self.fast_sims is not None:
            self._init_cap()

    def _init_endgame(self) -> None:
        Q, dev = self.endgame_cap, self.device
        H = Q * self.max_plies

        def e(n, dt):
            return torch.empty(n, dtype=dt, device=dev)

        self.eg_me, self.eg_opp = e(Q, torch.int64), e(Q, torch.int64)
        self.eg_player, self.eg_ply, self.eg_game_id, self.eg_row = (e(Q, torch.int8), e(Q, torch.int32),
                                                                     e(Q, torch.int64), e(Q, torch.int32))
        self.eg_hist_me, self.eg_hist_opp = e(H, torch.int64), e(H, torch.int64)
        self.eg_hist_player, self.eg_hist_action = e(H, torch.int8), e(H, torch.uint8)
        self.eg_hist_pi = e(H * N_ACTIONS, torch.float32)
        self.eg_count = torch.zeros(1, dtype=torch.int32, device=dev)
        self.eg_counters = torch.zeros(4, dtype=torch.int64, device=dev)
        self.eg_workspace = e(max(int(self._L.bz_selfplay_endgame_workspace_bytes(Q)), 16), torch.uint8)
        g = BzSelfplayEndgameState()
        g.empties, g.cap, g.max_plies = self.endgame_empties, Q, self.max_plies
        for name, _ in BzSelfplayEndgameState._fields_[BzSelfplayEndgameState.N_SCALARS:]:
            setattr(g, name, getattr(self, "eg_" + name).data_ptr())
        self.eg = g
        self._eg_ref = C.byref(g)

    def _init_resign(self, threshold: float) -> None:
        dev = self.device
        self.hist_q = torch.empty(max(self.n_games, 1) * self.max_plies, dtype=torch.float32, device=dev)
        self.eg_hist_q = (torch.empty(self.endgame_cap * self.max_plies, dtype=torch.float32, device=dev)
                          if self.eg is not None else None)
        self.rp_q = torch.empty(max(self.replay_cap, 1), dtype=torch.float32, device=dev)
        self.resign_counters = torch.zeros(2, dtype=torch.int64, device=dev)
        r = BzSelfplayResignState()
        r.threshold, r.audit_below = threshold, self._audit_below
        r.hist_q, r.rp_q, r.counters = self.hist_q.data_ptr(), self.rp_q.data_ptr(), self.resign_counters.data_ptr()
        r.eg_hist_q = self.eg_hist_q.data_ptr() if self.eg_hist_q is not None else None
        self.rs = r
        self._rs_ref = C.byref(r)

    def _init_cap(self) -> None:
        dev, T = self.device, self.pools.n_trees

        def e(n, dt):
            return torch.empty(max(n, 1), dtype=dt, device=dev)

        self.tree_of_slot = e(self.n_games, torch.int32)
        self.cap_root_me, self.cap_root_opp = e(T, torch.int64), e(T, torch.int64)
        self.pair_entrant = e(-(-T // PAIR_TREES), torch.uint8)
        self.hist_full = e(self.n_games * self.max_plies, torch.uint8)
        self.eg_hist_full = e(self.endgame_cap * self.max_plies, torch.uint8) if self.eg is not None else None
        self.rp_full = e(self.replay_cap, torch.uint8)
        self.cap_counters = torch.zeros(2, dtype=torch.int64, device=dev)
        c = BzSelfplayCapState()
        c.full_below, c.n_trees = self._full_below, T
        for name in ("tree_of_slot", "pair_entrant", "hist_full", "eg_hist_full", "rp_full"):
            t = getattr(self, name)
            setattr(c, name, t.data_ptr() if t is not None else None)
        c.root_me, c.root_opp, c.counters = (self.cap_root_me.data_ptr(), self.cap_root_opp.data_ptr(),
                                             self.cap_counters.data_ptr())
        self.cs = c
        self._cs_ref = C.byref(c)

    def _search_cap(self) -> None:
        """layout -> reset from the layout's roots -> the two budgets in one bz_mcts_search_fused_entrants; with root
        noise the first iteration runs through the per-iteration kernels and the noise goes to the full pairs only"""
        m, st = self.mcts, _lib.stream_ptr()
        _lib.check(self._L.bz_selfplay_cap_layout(self._ref, self._cs_ref, st), "bz_selfplay_cap_layout")
        self.launches += 1
        m.reset(self.cap_root_me, self.cap_root_opp)
        K = self.pools.n_leaves
        iters = [self.n_sims // K, self.fast_sims // K]
        if m.dirichlet_alpha > 0:
            m.select()
            m.evaluate()
            m.expand_backup()
            m.add_root_noise(self.pair_entrant, 0)
            iters = [n - 1 for n in iters]
        img = m.evaluator.net._image_pair.data_ptr()  # read at every ply: refresh() may rebuild the image
        _lib.check(self._L.bz_mcts_search_fused_entrants(self.pools._ref, (C.c_void_p * 2)(img, img),
                                                         (C.c_int32 * 2)(*iters), 2, _lib.dptr(self.pair_entrant), st),
                   "bz_mcts_search_fused_entrants")
        m.launches += -(-self.pools.n_trees // m.ONE_LAUNCH_MAX_TREES)  # one launch per chunk of <= 4144 trees

    @property
    def resign_threshold(self) -> float | None:
        """the threshold of the next plies (float32), None when resignation is off"""
        return None if self.rs is None else float(self.rs.threshold)

    def set_resign_threshold(self, v: float) -> None:
        """a new threshold in [-1, 1] for the following plies (resignation must have been switched on)"""
        if self.rs is None:
            raise RuntimeError("set_resign_threshold needs BatchedSelfPlay(resign_threshold=...)")
        self.rs.threshold = _resign.check_threshold(v)

    # -- one lockstep ply for every game ----------------------------------------------------------
    def search(self) -> None:
        if self.cs is not None:
            self._search_cap()
            self._moves += 1
            return
        if (self.mcts.use_graph and self.mcts._graph is None and not self.mcts.one_launch
                and self.n_sims // self.pools.n_leaves - 1 >= self.mcts.unroll):
            self.mcts.prepare()  # lazily, before the roots are set: play_move() works without an explicit prepare()
        if self.reuse and self._moves > 0:
            self.mcts.advance(self.last_action, self.me, self.opp)  # slots whose game restarted get an empty tree
        else:
            self.mcts.reset(self.me, self.opp)
        self.mcts.run(self.n_sims)
        self._moves += 1

    def advance(self) -> None:
        if self.cs is not None:
            _lib.check(self._L.bz_selfplay_advance_cap(self._ref, self._eg_ref if self.eg is not None else None,
                                                       self._rs_ref if self.rs is not None else None, self._cs_ref,
                                                       self.pools._ref, _lib.dptr(self.last_action), _lib.stream_ptr()),
                       "bz_selfplay_advance_cap")
            self.launches += 1
            if self.eg is not None:
                self._advances += 1
                if self._advances % self.endgame_every == 0:
                    self.endgame_play()
            return
        if self.rs is not None:
            _lib.check(self._L.bz_selfplay_advance_resign(self._ref, self._eg_ref if self.eg is not None else None,
                                                          self._rs_ref, self.pools._ref, _lib.dptr(self.last_action),
                                                          _lib.stream_ptr()), "bz_selfplay_advance_resign")
            self.launches += 1
            if self.eg is not None:
                self._advances += 1
                if self._advances % self.endgame_every == 0:
                    self.endgame_play()
            return
        if self.eg is None:
            _lib.check(self._L.bz_selfplay_advance(self._ref, self.pools._ref, _lib.dptr(self.last_action),
                                                   _lib.stream_ptr()), "bz_selfplay_advance")
            self.launches += 1
            return
        _lib.check(self._L.bz_selfplay_advance_endgame(self._ref, self._eg_ref, self.pools._ref, _lib.dptr(self.last_action),
                                                       _lib.stream_ptr()), "bz_selfplay_advance_endgame")
        self.launches += 1
        self._advances += 1
        if self._advances % self.endgame_every == 0:
            self.endgame_play()

    def endgame_play(self) -> None:
        """One solver phase: every game in the endgame queue is played to its end by the exact solver (or the
        win/draw/loss solver, ``endgame_solve="wld"``) and flushed to the replay buffer (a fixed number of launches, no
        host synchronisation).  ``advance`` calls it every ``endgame_every`` plies."""
        if self.eg is None:
            raise RuntimeError("endgame_play needs endgame_empties > 0")
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        if self.cs is not None:
            name = "bz_selfplay_endgame_play_cap"
            _lib.check(self._L.bz_selfplay_endgame_play_cap(self._ref, self._eg_ref, self._rs_ref if self.rs is not None
                                                            else None, self._cs_ref, _lib.dptr(self.eg_workspace),
                                                            int(self.endgame_solve == "wld"), _lib.stream_ptr()), name)
        elif self.rs is not None:
            name = "bz_selfplay_endgame_play_resign"
            _lib.check(self._L.bz_selfplay_endgame_play_resign(self._ref, self._eg_ref, self._rs_ref,
                                                               _lib.dptr(self.eg_workspace), int(self.endgame_solve == "wld"),
                                                               _lib.stream_ptr()), name)
        else:
            name = "bz_selfplay_endgame_play_wld" if self.endgame_solve == "wld" else "bz_selfplay_endgame_play"
            _lib.check(getattr(self._L, name)(self._ref, self._eg_ref, _lib.dptr(self.eg_workspace), _lib.stream_ptr()), name)
        t1.record()
        self._eg_events.append((t0, t1))
        self.launches += 6 * 2 * self.endgame_empties  # per solver ply: the solve's four kernels, the move, the compaction

    def endgame_ms(self) -> float:
        """milliseconds spent in solver phases so far (CUDA events; waits for the phases recorded since the last call)"""
        for t0, t1 in self._eg_events:
            t1.synchronize()
            self._eg_ms += t0.elapsed_time(t1)
        self._eg_events = []
        return self._eg_ms

    def play_move(self) -> None:
        self.search()
        self.advance()

    def prepare(self) -> None:
        """capture the CUDA graph (before the first search); randomized budgets run the one-launch search, no graph"""
        if self.cs is None:
            self.mcts.prepare()

    # -- results ---------------------------------------------------------------------------------
    def stats(self) -> dict:
        c = self.counters.cpu().tolist()
        out = {"replay_records": c[0], "plies": c[1], "o_wins": c[2], "draws": c[3], "x_wins": c[4],
               "dropped": c[5], "games": c[6]}
        # endgame handover: games the solver finished, plies it played, games waiting in the queue, handovers refused
        # because the queue was full (those games are searched to their end in their slots)
        eg = self.eg_counters.cpu().tolist() if self.eg is not None else [0, 0, 0, 0]
        out.update({"endgame_games": eg[3], "endgame_plies": eg[1],
                    "endgame_pending": int(self.eg_count.item()) if self.eg is not None else 0, "endgame_overflow": eg[2]})
        # resignation: games resigned, audited games finished (both 0 when it is off)
        rc = self.resign_counters.cpu().tolist() if self.rs is not None else [0, 0]
        out.update({"resigned": rc[0], "audited": rc[1]})
        # randomized budgets: searched plies with the full budget and with the fast one (both 0 when it is off)
        cc = self.cap_counters.cpu().tolist() if self.cs is not None else [0, 0]
        out.update({"full_plies": cc[0], "fast_plies": cc[1]})
        return out

    def drain_replay(self) -> dict:
        """Returns the finished games' records (device tensors, copies) and empties the buffer.  Games in the endgame
        queue are games in progress, like those in the slots: a later solver phase finishes them."""
        c = self.counters.cpu().tolist()
        n = min(int(c[0]), self.replay_cap)  # counters[0] counts committed rows only (a game that does not fit takes none)
        if c[5] > self._dropped_seen:
            import warnings

            warnings.warn(f"replay buffer overflow: {c[5] - self._dropped_seen} records of finished games were dropped "
                          f"(replay_cap {self.replay_cap}); drain more often or enlarge replay_cap", RuntimeWarning)
            self._dropped_seen = c[5]
        out = {
            "me": self.rp_me[:n].clone(), "opp": self.rp_opp[:n].clone(),
            "pi": self.rp_pi[: n * N_ACTIONS].view(n, N_ACTIONS).clone(),
            "z": self.rp_z[:n].clone(), "game": self.rp_game[:n].clone(), "ply": self.rp_ply[:n].clone(),
        }
        if self.rs is not None:
            out["q"] = self.rp_q[:n].clone()  # q of the record's ply (NaN for solver-played plies)
        if self.cs is not None:
            out["full"] = self.rp_full[:n].clone()  # 1: a full search's (or the solver's) pi; 0: a fast search's
        self.counters[0] = 0
        return out

    def total_launches(self) -> int:
        return self.launches + self.mcts.launches
