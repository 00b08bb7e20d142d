"""Batched MCTS host side: tree pools in HBM + the lockstep search loop (kernels K5-K8).

The reference has no MCTS (SURVEY.md section 0.2); the search serves its
``Player.get_move(board) -> (row, col)`` contract (reversi_players.py:5-8, players.py:6-9) and
follows the semantics frozen in oracle/mcts_ref.py.  One search of ``n_sims`` iterations is

    reset -> select -> [evaluate -> step]*(n_sims-1) -> evaluate -> expand_backup

where ``step`` = expand+backup of iteration i fused with the select+gather of iteration i+1 in
ONE kernel launch, and ``[evaluate -> step]`` blocks are replayed from a CUDA graph.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from ._lib import BzTreePools

GAME_REVERSI, GAME_TTT = 0, 1
LEAF_EVAL, LEAF_TERMINAL, LEAF_ERROR = 0, 1, 2
PRIOR_WEIGHTS, PRIOR_LOGITS_BF16 = 0, 1
MAX_ARENA_UNITS = 0x7FFF0
_NODE_UNITS = {GAME_REVERSI: 18, GAME_TTT: 6}  # worst-case node block: 33 (8x8 Reversi) / 9 edges


class TreePools:
    """Caller-owned pools for ``n_trees`` concurrent trees (``bz_tree_pools``): one arena of node
    blocks per tree plus the per-tree pending-leaf records, all resident in HBM.

    ``sims_cap``: the largest number of iterations a search will run between resets; every
    iteration expands at most one node and a node block takes at most 18 (Reversi) / 6 (TTT)
    32-byte units, so ``arena_units = sims_cap * that`` can never overflow.  A smaller
    ``arena_units`` may be passed (mean branching is ~8-10); overflow is detected and raised,
    never silent.
    """

    def __init__(self, n_trees: int, sims_cap: int, game: int = GAME_REVERSI, board_size: int = 8,
                 c_puct: float = 1.25, arena_units: int | None = None, max_depth: int | None = None,
                 prior_mode: int = PRIOR_WEIGHTS, eval_stride: int = 0, group_lanes: int = 0, n_leaves: int = 1,
                 device="cuda", reuse: bool = False):
        if game not in (GAME_REVERSI, GAME_TTT):
            raise ValueError("game must be GAME_REVERSI or GAME_TTT")
        self.game, self.board_size = game, (3 if game == GAME_TTT else board_size)
        self.n_trees, self.sims_cap = int(n_trees), int(sims_cap)
        self.n_actions = 9 if game == GAME_TTT else 65
        self.c_puct = float(c_puct)
        # reuse: the trees may be kept across moves (BatchedMCTS.advance / bz_mcts_reroot).  The arena then holds the
        # kept subtree AND the worst case of the next search: twice the default size, and a subtree is only kept if it
        # leaves room for sims_cap worst-case nodes (reuse_cap_units), so a search still cannot overflow the arena.
        self.reuse = bool(reuse)
        worst = max(self.sims_cap, 1) * _NODE_UNITS[game]
        if arena_units is None:
            arena_units = min(worst * (2 if self.reuse else 1), MAX_ARENA_UNITS)
        arena_units = max(int(arena_units), 18)
        if arena_units > MAX_ARENA_UNITS:
            raise ValueError(f"arena_units {arena_units} exceeds {MAX_ARENA_UNITS}")
        self.arena_units = arena_units
        self.reuse_cap_units = max(arena_units - worst, 0)
        self.max_depth = int(max_depth or (16 if game == GAME_TTT else 128))
        self.prior_mode, self.eval_stride = int(prior_mode), int(eval_stride)
        self.device = torch.device(device)
        # leaves per tree and iteration: 1 = the sequential parity definition; K > 1 = K descents with virtual loss
        # (oracle/mcts_ref.py MCTS.select_vl).  Pending-leaf arrays are slot-major: row = slot * n_trees + tree.
        if not 1 <= int(n_leaves) <= 8:
            raise ValueError("n_leaves must be in 1..8")
        self.n_leaves = int(n_leaves)
        self.n_rows = self.n_trees * self.n_leaves
        B = max(self.n_trees, 1)
        R = max(self.n_rows, 1)
        dev = self.device

        def e(n, dt):
            return torch.empty(max(n, 1), dtype=dt, device=dev)

        self.root_me, self.root_opp = e(B, torch.int64), e(B, torch.int64)
        # valid "empty tree" state from the start, so no kernel ever walks uninitialised memory
        self.root_meta = torch.full((B,), -8192, dtype=torch.int32, device=dev)  # meta(UNEXPANDED)
        self.arena_used = torch.zeros(B, dtype=torch.int32, device=dev)
        self.edge_count, self.sim_count = torch.zeros(B, dtype=torch.int32, device=dev), e(B, torch.int32)
        self.depth_sum, self.error = e(B, torch.int32), torch.zeros(B, dtype=torch.int32, device=dev)
        self.arena = e(B * self.arena_units * 8, torch.int32)
        # scratch of bz_mcts_reroot (the subtree is compacted there and copied back) + the visits every root inherited
        self.scratch = e(B * self.arena_units * 8, torch.int32) if self.reuse else None
        self.inherited = torch.zeros(B, dtype=torch.int32, device=dev)
        self.path, self.path_len = e(R * self.max_depth * 4, torch.int32), torch.zeros(R, dtype=torch.int32, device=dev)
        self.leaf_parent = e(R, torch.int32)
        self.leaf_me, self.leaf_opp, self.leaf_mask = e(R, torch.int64), e(R, torch.int64), e(R, torch.int64)
        self.leaf_status = torch.full((R,), LEAF_ERROR, dtype=torch.uint8, device=dev)
        self.leaf_action = e(R, torch.uint8)
        self.leaf_value = e(R, torch.float32)
        if game == GAME_TTT:
            self.leaf_planes = torch.zeros((R, 9), dtype=torch.bfloat16, device=dev)
        else:
            self.leaf_planes = torch.zeros((R, 2, 8, 8), dtype=torch.bfloat16, device=dev)
        s = BzTreePools()
        s.game, s.board_size, s.n_trees, s.n_actions = game, (self.board_size if game == GAME_REVERSI else 8), self.n_trees, self.n_actions
        s.arena_units, s.max_depth, s.c_puct, s.prior_mode = self.arena_units, self.max_depth, self.c_puct, self.prior_mode
        if group_lanes not in (0, 8, 16, 32):
            raise ValueError("group_lanes must be 0 (auto), 8, 16 or 32")
        self.group_lanes = int(group_lanes)
        s.eval_stride, s.group_lanes = self.eval_stride, self.group_lanes
        s.n_leaves = self.n_leaves
        for name, _ in BzTreePools._fields_[BzTreePools.N_SCALARS:]:
            setattr(s, name, getattr(self, name).data_ptr())
        self.c_struct = s
        self._ref = C.byref(s)

    def set_prior_mode(self, mode: int, eval_stride: int = 0) -> None:
        self.prior_mode, self.eval_stride = int(mode), int(eval_stride)
        self.c_struct.prior_mode, self.c_struct.eval_stride = self.prior_mode, self.eval_stride

    # bytes of HBM held by the pools
    def nbytes(self) -> int:
        return sum(getattr(self, n).numel() * getattr(self, n).element_size()
                   for n, _ in BzTreePools._fields_[BzTreePools.N_SCALARS:])


class HashEvaluator:
    """Parity-mode evaluator: the integer-hash pseudo-net (``bz_hash_eval``), exact in fp32 and
    identical to oracle/mcts_ref.py:hash_eval.  Produces prior WEIGHTS (BZ_PRIOR_WEIGHTS)."""

    prior_mode = PRIOR_WEIGHTS

    def __init__(self, salt: int = 0):
        self.salt = int(salt)

    def bind(self, pools: "TreePools"):
        B, A = max(pools.n_rows, 1), pools.n_actions  # one row per pending leaf
        self.out = torch.zeros((B, A), dtype=torch.float32, device=pools.device)
        self.value = torch.zeros(B, dtype=torch.float32, device=pools.device)
        return self.out, self.value

    def __call__(self, pools: "TreePools") -> None:
        L = _lib.load()
        _lib.check(L.bz_hash_eval(_lib.dptr(pools.leaf_me), _lib.dptr(pools.leaf_opp), self.salt, pools.n_actions,
                                  _lib.dptr(self.out), _lib.dptr(self.value), pools.n_rows, _lib.stream_ptr()),
                   "bz_hash_eval")


class WeightsEvaluator:
    """Evaluator fed from outside (tests / replaying recorded priors): fill ``out`` and ``value``."""

    prior_mode = PRIOR_WEIGHTS

    def bind(self, pools: "TreePools"):
        B, A = max(pools.n_rows, 1), pools.n_actions  # one row per pending leaf
        self.out = torch.zeros((B, A), dtype=torch.float32, device=pools.device)
        self.value = torch.zeros(B, dtype=torch.float32, device=pools.device)
        return self.out, self.value

    def __call__(self, pools: "TreePools") -> None:
        pass


class NetEvaluator:
    """PyTorch policy/value net on the gathered bf16 leaf planes, parity-friendly form: the net
    returns ``(logits [B, A], value [B])``, prior weights are ``softmax(logits)`` in fp32 and the
    tree kernel renormalises them over the legal actions (BZ_PRIOR_WEIGHTS).  The weights of a
    search can be recorded and replayed into the oracle."""

    prior_mode = PRIOR_WEIGHTS

    def __init__(self, net: torch.nn.Module):
        self.net = net

    def bind(self, pools: "TreePools"):
        B, A = max(pools.n_rows, 1), pools.n_actions  # one row per pending leaf
        self.out = torch.zeros((B, A), dtype=torch.float32, device=pools.device)
        self.value = torch.zeros(B, dtype=torch.float32, device=pools.device)
        return self.out, self.value

    @torch.no_grad()
    def __call__(self, pools: "TreePools") -> None:
        logits, value = self.net(pools.leaf_planes)
        torch.softmax(logits.float(), dim=-1, out=self.out)
        self.value.copy_(value.reshape(-1))


class FusedNetEvaluator:
    """Throughput form: the net's ``forward_raw(planes) -> bf16 [B, stride]`` (policy logits in
    columns 0..A-1, pre-tanh value in column A) is handed to the tree kernel as is; the kernel does
    the legal-move softmax and the tanh itself (BZ_PRIOR_LOGITS_BF16), so an iteration is the net's
    GEMMs plus ONE tree kernel."""

    prior_mode = PRIOR_LOGITS_BF16

    def __init__(self, net: torch.nn.Module, use_kernel: bool | str | None = None, pdl: bool | None = None):
        if not hasattr(net, "forward_raw"):
            raise TypeError("FusedNetEvaluator needs a net with forward_raw()")
        self.net = net
        # None: the single-launch tcgen05 MLP kernels (bz_mlp_forward_pair / _pair2) when the shape allows, else
        # the library GEMMs; True / "pair" / "pair2" / False force one path
        self.use_kernel = use_kernel
        # programmatic dependent launch between the MLP kernel and the tree step kernel (process-wide
        # switch, results identical): on by default whenever the kernel path may be taken
        self.pdl = (use_kernel is not False) if pdl is None else bool(pdl)

    def bind(self, pools: "TreePools"):
        B = max(pools.n_rows, 1)  # one row per pending leaf
        self.stride = int(self.net.raw_width)
        self.out = torch.zeros((B, self.stride), dtype=torch.bfloat16, device=pools.device)
        self.value = torch.zeros(1, dtype=torch.float32, device=pools.device)  # unused in this mode
        pools.set_prior_mode(PRIOR_LOGITS_BF16, self.stride)
        self.refresh()
        # 1 when the forward is one kernel of libbetazero_b200 (bench.py's gpu_launches), 0 for library GEMMs
        k = self.use_kernel
        if k is None:
            k = hasattr(self.net, "fused_kernel_ok") and self.net.fused_kernel_ok(pools.leaf_planes)
        self.own_launches = 1 if k else 0
        return self.out, self.value

    def refresh(self) -> None:
        """rebuild the net's fused inference weights (after a weight update / broadcast)"""
        if hasattr(self.net, "prepare_inference"):
            self.net.prepare_inference()

    @torch.no_grad()
    def __call__(self, pools: "TreePools") -> None:
        self.net.forward_raw(pools.leaf_planes, out=self.out, fused=self.use_kernel)


class BatchedMCTS:
    """Lockstep search over all trees of a :class:`TreePools`.

    ``evaluator.bind(pools)`` returns the (eval_out, value) buffers the tree kernels read;
    ``evaluator(pools)`` must be stream-ordered GPU work that reads ``pools.leaf_planes`` (or
    ``leaf_me/leaf_opp``) and fills them; it is captured into the CUDA graph with the tree kernel.
    """

    def __init__(self, pools: TreePools, evaluator, use_graph: bool = True, graph_unroll: int = 16, fused: bool = True,
                 dirichlet_alpha: float = 0.0, dirichlet_eps: float = 0.25, noise_seed: int = 0,
                 one_launch: bool | None = None):
        self.pools, self.evaluator = pools, evaluator
        # one_launch: run the whole search of a move in ONE kernel (bz_mcts_search_fused) when the shape allows --
        # Reversi, one leaf per iteration or 2 / 4 in wave mode, the bf16 MLP through its tcgen05 kernel path (more than 4144
        # trees are searched in chunks, one launch each).
        # None = whenever possible; False = always the per-iteration kernels; True = raise if the shape does not fit.
        self._one_launch_arg = one_launch
        # root exploration noise (self-play only; 0 = off, which every parity test uses)
        self.dirichlet_alpha, self.dirichlet_eps = float(dirichlet_alpha), float(dirichlet_eps)
        self._noise_gen = torch.Generator(device=pools.device).manual_seed(int(noise_seed)) if dirichlet_alpha > 0 else None
        self.use_graph, self.unroll, self.fused = bool(use_graph), int(graph_unroll), bool(fused)
        B, A = max(pools.n_trees, 1), pools.n_actions
        if evaluator is None:
            evaluator = self.evaluator = WeightsEvaluator()
        self.prior_w, self.value = evaluator.bind(pools)  # eval_out / value buffers the kernels read
        pools.set_prior_mode(evaluator.prior_mode, getattr(evaluator, "stride", 0))
        self.counts = torch.zeros((B, A), dtype=torch.int32, device=pools.device)
        self.pi = torch.zeros((B, A), dtype=torch.float32, device=pools.device)
        self.q = torch.zeros((B, A), dtype=torch.float32, device=pools.device)
        self.best = torch.zeros(B, dtype=torch.uint8, device=pools.device)
        self._graph = None
        self._L = _lib.load()
        self.launches = 0  # kernels of libbetazero_b200 launched (bench.py's gpu_launches)
        # Programmatic dependent launch is a property of THIS search's kernel sequence: only an evaluator that puts a
        # kernel between two step kernels (FusedNetEvaluator) may ask for it; applied before every launch / capture.
        self._pdl = bool(getattr(evaluator, "pdl", False))

    # -- the one-launch search ------------------------------------------------------------------
    ONE_LAUNCH_MAX_TREES = 148 * 28

    def one_launch_ok(self) -> bool:
        """bz_mcts_search_fused covers this search (same trees, bit for bit, as the per-iteration kernels)."""
        p, ev = self.pools, self.evaluator
        net = getattr(ev, "net", None)
        return (isinstance(ev, FusedNetEvaluator) and ev.use_kernel is not False and getattr(ev, "own_launches", 0) == 1
                and getattr(net, "_image_pair", None) is not None and self.fused
                and p.game == GAME_REVERSI and ((p.n_leaves in (2, 4) and p.group_lanes in (0, 32)) or p.n_leaves == 1)
                and p.prior_mode == PRIOR_LOGITS_BF16 and p.eval_stride == 72 and p.n_trees > 0)

    @property
    def one_launch(self) -> bool:
        if self._one_launch_arg is False:
            return False
        ok = self.one_launch_ok()
        if self._one_launch_arg is None and ok and self.pools.n_leaves == 1 and self.pools.n_trees > self.ONE_LAUNCH_MAX_TREES:
            # one leaf per iteration and more trees than one launch holds: the per-iteration kernels with 16 / 8 lanes per
            # tree fill the GPU better than chunks of 4144 one after the other (65 536 trees: 776 M against ~320 M sims/s)
            return False
        if self._one_launch_arg and not ok:
            raise RuntimeError("one_launch=True, but bz_mcts_search_fused does not cover this search (it needs Reversi, "
                               "n_leaves = 1 or n_leaves = 2 / 4 in wave mode, and the bf16 MLP kernel path)")
        return ok

    def search_one_launch(self, n_iterations: int) -> None:
        """select, then n_iterations x [net, expand + backup, select (not after the last)] in one kernel."""
        _lib.check(self._L.bz_mcts_search_fused(self.pools._ref, _lib.dptr(self.evaluator.net._image_pair),
                                                _lib.dptr(self.prior_w), int(n_iterations), _lib.stream_ptr()),
                   "bz_mcts_search_fused")
        self.launches += -(-self.pools.n_trees // self.ONE_LAUNCH_MAX_TREES)  # one launch per chunk of <= 4144 trees

    # -- single kernels ------------------------------------------------------------------------
    def reset(self, root_me: torch.Tensor, root_opp: torch.Tensor) -> None:
        p = self.pools
        if root_me.numel() != p.n_trees or root_opp.numel() != p.n_trees:
            raise ValueError("one root per tree expected")
        _lib.check(self._L.bz_mcts_reset(p._ref, _lib.dptr(root_me), _lib.dptr(root_opp), _lib.stream_ptr()), "bz_mcts_reset")
        p.inherited.zero_()
        self.launches += 1

    def select(self) -> None:
        _lib.set_pdl(self._pdl)
        _lib.check(self._L.bz_mcts_select(self.pools._ref, _lib.stream_ptr()), "bz_mcts_select")
        self.launches += 1

    def evaluate(self) -> None:
        _lib.set_pdl(self._pdl)
        self.evaluator(self.pools)
        self.launches += getattr(self.evaluator, "own_launches", 0)  # kernels of this library the evaluator launched

    def expand_backup(self) -> None:
        _lib.set_pdl(self._pdl)
        _lib.check(self._L.bz_mcts_expand_backup(self.pools._ref, _lib.dptr(self.prior_w), _lib.dptr(self.value),
                                                 _lib.stream_ptr()), "bz_mcts_expand_backup")
        self.launches += 1

    def step(self) -> None:
        if self.fused:
            _lib.set_pdl(self._pdl)
            _lib.check(self._L.bz_mcts_step(self.pools._ref, _lib.dptr(self.prior_w), _lib.dptr(self.value),
                                            _lib.stream_ptr()), "bz_mcts_step")
            self.launches += 1
        else:
            self.expand_backup()
            self.select()

    # -- the search ----------------------------------------------------------------------------
    def _capture(self) -> None:
        # warm up on a side stream (cuBLAS workspaces, lazy module init), then capture `unroll`
        # [evaluate -> step] blocks.  The warm-up really runs, so the pools must hold valid trees:
        # reset them to start positions first (the caller resets again for the real search).
        p = self.pools
        if p.game == GAME_TTT:
            rm = torch.zeros(p.n_trees, dtype=torch.int64, device=p.device)
            ro = torch.zeros_like(rm)
        else:
            from . import env

            rm, ro, _ = env.reversi_init(p.n_trees, p.board_size, device=p.device)
        self.reset(rm, ro)
        self.select()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(2):
                self.evaluate()
                self.step()
        torch.cuda.current_stream().wait_stream(s)
        g = torch.cuda.CUDAGraph()
        n0 = self.launches
        with torch.cuda.graph(g):
            for _ in range(self.unroll):
                self.evaluate()
                self.step()
        self._graph_launches = self.launches - n0
        self._graph = g

    def run(self, n_sims: int) -> None:
        """n_sims simulations on the current trees (after :meth:`reset`): n_sims / n_leaves iterations."""
        if n_sims <= 0:
            return
        if n_sims > self.pools.sims_cap:
            raise ValueError(f"n_sims {n_sims} exceeds the pools' sims_cap {self.pools.sims_cap}")
        K = self.pools.n_leaves
        if n_sims % K:
            raise ValueError(f"n_sims {n_sims} is not a multiple of the pools' n_leaves {K}")
        if self.pools.n_trees == 0:
            return
        inner = n_sims // K - 1
        if self.one_launch:
            if self.dirichlet_alpha > 0:
                if inner == 0:
                    raise ValueError(f"dirichlet_alpha > 0 needs at least two iterations (n_sims >= {2 * K}); got n_sims = {n_sims}")
                # iteration 1 expands the root with the per-iteration kernels; its priors are perturbed before the rest
                self.select()
                self.evaluate()
                self.expand_backup()
                self.add_root_noise()
                self.search_one_launch(inner)
            else:
                self.search_one_launch(inner + 1)
            return
        if self.dirichlet_alpha > 0 and inner == 0:
            # the noise perturbs the priors of the root that iteration 1 expands: a one-iteration search never uses it
            raise ValueError(f"dirichlet_alpha > 0 needs at least two iterations (n_sims >= {2 * K}); got n_sims = {n_sims}")
        if self.use_graph and self._graph is None and inner - (1 if self.dirichlet_alpha > 0 else 0) >= self.unroll:
            raise RuntimeError("the CUDA graph is captured by prepare() (or search()) BEFORE reset(): capturing runs warm-up "
                               "iterations on the pools and would clobber the roots just set")
        self.select()
        if self.dirichlet_alpha > 0 and inner > 0:
            # iteration 1 expands the root; perturb its priors before the second descent
            self.evaluate()
            self.expand_backup()
            self.add_root_noise()
            self.select()
            inner -= 1
        if self.use_graph and inner >= self.unroll:
            for _ in range(inner // self.unroll):
                self._graph.replay()
                self.launches += self._graph_launches
            inner %= self.unroll
        for _ in range(inner):
            self.evaluate()
            self.step()
        self.evaluate()
        self.expand_backup()

    def add_root_noise(self, pair_entrant: torch.Tensor | None = None, entrant: int = 0) -> None:
        """P_root <- (1 - eps) P + eps Dirichlet(alpha) over the root's legal moves (bz_mcts_root_noise).
        Gamma(alpha, 1) samples come from torch (plumbing); the kernel normalises over the legal edges.  With
        ``pair_entrant`` (uint8 per CTA pair of 56 trees) only the trees of the pairs of ``entrant`` get the noise
        (bz_mcts_root_noise_entrant)."""
        p = self.pools
        shape = (max(p.n_trees, 1), p.n_actions)
        alpha = torch.full(shape, self.dirichlet_alpha, dtype=torch.float32, device=p.device)
        noise = torch._standard_gamma(alpha, generator=self._noise_gen).clamp_min_(1e-30)
        if pair_entrant is None:
            _lib.check(self._L.bz_mcts_root_noise(p._ref, _lib.dptr(noise), self.dirichlet_eps, _lib.stream_ptr()),
                       "bz_mcts_root_noise")
        else:
            _lib.check(self._L.bz_mcts_root_noise_entrant(p._ref, _lib.dptr(noise), self.dirichlet_eps,
                                                          _lib.dptr(pair_entrant), int(entrant), _lib.stream_ptr()),
                       "bz_mcts_root_noise_entrant")
        self.launches += 1

    def prepare(self) -> None:
        """Capture the CUDA graph (clobbers the pending leaf state: call before reset())."""
        if self.use_graph and self._graph is None and self.pools.n_trees > 0 and not self.one_launch:
            self._capture()

    def search(self, root_me: torch.Tensor, root_opp: torch.Tensor, n_sims: int, check: bool = True):
        """Fresh search from the given roots.  Returns (visit_counts, pi, q) device tensors."""
        if self.use_graph and self._graph is None and n_sims // self.pools.n_leaves - 1 >= self.unroll and not self.one_launch:
            self.prepare()
        self.reset(root_me, root_opp)
        self.run(n_sims)
        out = self.root_policy()
        if check:
            self.check_errors()
        return out

    def search_host(self, root_me: torch.Tensor, root_opp: torch.Tensor, n_sims: int):
        """The host-facing form of :meth:`search` (``Player.get_move`` for a batch of boards that live in HOST memory):
        roots from host tensors -> pinned staging -> H2D -> fresh search -> pi + most visited action -> D2H, one stream
        synchronisation.  Returns ``(pi float32 [B, A], action uint8 [B])`` as pinned host tensors that stay valid until the
        next call.  With the one-launch search (and no root noise) the whole sequence -- copies, reset, search, policy
        kernels -- is captured once in a CUDA graph and replayed: one launch from the host per call instead of eight."""
        p = self.pools
        B, A = max(p.n_trees, 1), p.n_actions
        if root_me.numel() != p.n_trees or root_opp.numel() != p.n_trees:
            raise ValueError("one root per tree expected")
        st = getattr(self, "_host", None)
        if st is None:
            st = self._host = {
                "h_me": torch.empty(B, dtype=torch.int64).pin_memory(), "h_opp": torch.empty(B, dtype=torch.int64).pin_memory(),
                "d_me": torch.empty(B, dtype=torch.int64, device=p.device), "d_opp": torch.empty(B, dtype=torch.int64, device=p.device),
                "h_pi": torch.empty((B, A), dtype=torch.float32).pin_memory(), "h_act": torch.empty(B, dtype=torch.uint8).pin_memory(),
                "graphs": {}}
        st["h_me"][: p.n_trees].copy_(root_me.reshape(-1))
        st["h_opp"][: p.n_trees].copy_(root_opp.reshape(-1))

        def body():
            st["d_me"].copy_(st["h_me"], non_blocking=True)
            st["d_opp"].copy_(st["h_opp"], non_blocking=True)
            self.reset(st["d_me"][: p.n_trees], st["d_opp"][: p.n_trees])
            self.run(n_sims)
            _, pi, _ = self.root_policy()
            act = self.best_action()
            st["h_pi"].copy_(pi, non_blocking=True)
            st["h_act"].copy_(act, non_blocking=True)

        if self.one_launch and self.dirichlet_alpha == 0 and p.n_trees > 0:
            g = st["graphs"].get(n_sims)
            if g is None:
                n0 = self.launches
                body()  # once eagerly: lazy initialisation (sqrt table, shared-memory opt-in) must not happen under capture
                torch.cuda.current_stream().synchronize()
                per_call = self.launches - n0
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    body()
                self.launches = n0
                st["graphs"][n_sims] = (g, per_call)
                g = st["graphs"][n_sims]
            g[0].replay()
            self.launches += g[1]
        else:
            body()
        torch.cuda.current_stream().synchronize()
        self.check_errors()
        return st["h_pi"], st["h_act"]

    def root_policy(self):
        p = self.pools
        _lib.check(self._L.bz_mcts_root_policy(p._ref, _lib.dptr(self.counts), _lib.dptr(self.pi), _lib.dptr(self.q),
                                               _lib.stream_ptr()), "bz_mcts_root_policy")
        self.launches += 1
        return self.counts, self.pi, self.q

    def best_action(self) -> torch.Tensor:
        _lib.check(self._L.bz_mcts_best_action(self.pools._ref, _lib.dptr(self.best), _lib.stream_ptr()),
                   "bz_mcts_best_action")
        self.launches += 1
        return self.best

    def check_errors(self) -> None:
        err = self.pools.error[: self.pools.n_trees]
        if self.pools.n_trees and bool(err.any().item()):
            codes = sorted(set(err[err != 0].tolist()))
            raise _lib.BzError(f"tree pool overflow (codes {codes}: 1 = arena, 2 = path depth); "
                               "enlarge arena_units / max_depth")

    def advance(self, action: torch.Tensor, root_me: torch.Tensor, root_opp: torch.Tensor, cap_units: int | None = None) -> None:
        """Tree reuse (opt-in, ``TreePools(reuse=True)``): the game of tree t has played ``action[t]`` and stands at
        ``(root_me[t], root_opp[t])``; every tree is re-rooted at the child that move leads to (bz_mcts_reroot) -- or
        emptied at the new position if that child was never expanded, is another position (a new game) or its subtree
        is larger than ``cap_units`` (default: what leaves room for a whole worst-case search).  The next ``run(n)``
        adds n simulations to the kept statistics.  Definition: oracle/mcts_ref.py MCTS.advance."""
        p = self.pools
        if p.scratch is None:
            raise RuntimeError("tree reuse needs TreePools(reuse=True) (a scratch arena and room for the kept subtree)")
        if action.numel() != p.n_trees or root_me.numel() != p.n_trees or root_opp.numel() != p.n_trees:
            raise ValueError("one action and one position per tree expected")
        if action.dtype != torch.uint8:
            raise TypeError("action: uint8 tensor expected")
        cap = p.reuse_cap_units if cap_units is None else int(cap_units)
        _lib.check(self._L.bz_mcts_reroot(p._ref, _lib.dptr(p.scratch), _lib.dptr(action), _lib.dptr(root_me), _lib.dptr(root_opp),
                                          cap, _lib.dptr(p.inherited), _lib.stream_ptr()), "bz_mcts_reroot")
        self.launches += 1

    def stats(self) -> dict:
        """mean path depth d and mean edges per expanded node b of the last search (roofline model)."""
        p = self.pools
        sims = int(p.sim_count[: p.n_trees].sum().item()) - int(p.inherited[: p.n_trees].sum().item())
        depth = int(p.depth_sum[: p.n_trees].sum().item())
        edges = int(p.edge_count[: p.n_trees].sum().item())
        units = int(p.arena_used[: p.n_trees].sum().item())
        return {"sims": sims, "mean_depth": depth / max(sims, 1), "edges": edges, "arena_units": units}

    def root_edges(self):
        """(N int32, W float32, P float32) of the root edges scattered by action, [B, A] each."""
        p = self.pools
        B, A = max(p.n_trees, 1), p.n_actions
        N = torch.zeros((B, A), dtype=torch.int32, device=p.device)
        W = torch.zeros((B, A), dtype=torch.float32, device=p.device)
        P = torch.zeros((B, A), dtype=torch.float32, device=p.device)
        _lib.check(self._L.bz_mcts_root_edges(p._ref, _lib.dptr(N), _lib.dptr(W), _lib.dptr(P), _lib.stream_ptr()),
                   "bz_mcts_root_edges")
        self.launches += 1
        return N, W, P
