"""ctypes binding of libbetazero_b200.so -- the only way this package computes anything.

There is NO CPU fallback: if the CUDA library is missing and cannot be built, importing a
compute path raises.  Device pointers are ``tensor.data_ptr()`` of CUDA tensors; the stream is
``torch.cuda.current_stream().cuda_stream`` (PyTorch is plumbing: device memory and streams).
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

_lib = None

ptr = C.c_void_p


class BzTreePools(C.Structure):
    """Mirror of ``bz_tree_pools`` (include/betazero_b200.h)."""

    _fields_ = [
        ("game", C.c_int32), ("board_size", C.c_int32), ("n_trees", C.c_int32), ("n_actions", C.c_int32),
        ("arena_units", C.c_int32), ("max_depth", C.c_int32), ("c_puct", C.c_float), ("prior_mode", C.c_int32),
        ("eval_stride", C.c_int32), ("group_lanes", C.c_int32), ("n_leaves", C.c_int32),
        ("root_me", ptr), ("root_opp", ptr), ("root_meta", ptr), ("arena_used", ptr), ("edge_count", ptr),
        ("sim_count", ptr), ("depth_sum", ptr), ("error", ptr),
        ("arena", ptr),
        ("path", ptr), ("path_len", ptr), ("leaf_parent", ptr), ("leaf_me", ptr), ("leaf_opp", ptr),
        ("leaf_mask", ptr), ("leaf_status", ptr), ("leaf_action", ptr), ("leaf_value", ptr), ("leaf_planes", ptr),
    ]
    N_SCALARS = 11


class BzSelfplayState(C.Structure):
    """Mirror of ``bz_selfplay_state`` (include/betazero_b200.h)."""

    _fields_ = [
        ("n_games", C.c_int32), ("board_size", C.c_int32), ("max_plies", C.c_int32), ("temp_plies", C.c_int32),
        ("seed", C.c_uint64), ("id_stride", C.c_int64), ("replay_cap", C.c_int64),
        ("me", ptr), ("opp", ptr), ("player", ptr), ("ply", ptr), ("game_id", ptr),
        ("hist_me", ptr), ("hist_opp", ptr), ("hist_player", ptr), ("hist_action", ptr), ("hist_pi", ptr),
        ("rp_me", ptr), ("rp_opp", ptr), ("rp_pi", ptr), ("rp_z", ptr), ("rp_game", ptr), ("rp_ply", ptr),
        ("counters", ptr),
    ]


class BzMatchState(C.Structure):
    """Mirror of ``bz_match_state`` (include/betazero_b200.h)."""

    _fields_ = [
        ("n_games", C.c_int32), ("board_size", C.c_int32), ("opening_plies", C.c_int32), ("n_trees", C.c_int32),
        ("seed", C.c_uint64), ("first_pair_id", C.c_int64),
        ("me", ptr), ("opp", ptr), ("player", ptr), ("ply", ptr), ("result", ptr), ("count_x", ptr), ("count_o", ptr),
        ("moves", ptr), ("tree_of_game", ptr),
        ("game_of_tree", ptr), ("root_me", ptr), ("root_opp", ptr), ("pair_net", ptr),
        ("counters", ptr),
    ]
    N_SCALARS = 6


class BzTournamentState(C.Structure):
    """Mirror of ``bz_tournament_state`` (include/betazero_b200.h)."""

    _fields_ = [("match", BzMatchState), ("n_entrants", C.c_int32), ("first", ptr), ("second", ptr)]


# name -> argtypes; every function returns int.  Must list EVERY symbol of include/betazero_b200.h
# (tests/test_abi.py cross-checks this table against the header).
_I64, _INT, _U64, _F = C.c_int64, C.c_int, C.c_uint64, C.c_float
_PP = C.POINTER(BzTreePools)
_SP = C.POINTER(BzSelfplayState)
_MP = C.POINTER(BzMatchState)
_TP = C.POINTER(BzTournamentState)
SIGNATURES = {
    "bz_abi_version": [],
    "bz_error_string": [_INT],
    "bz_set_pdl": [_INT],
    "bz_reversi_init": [ptr, ptr, ptr, _I64, _INT, ptr],
    "bz_reversi_legal_mask": [ptr, ptr, ptr, _I64, _INT, ptr],
    "bz_reversi_apply": [ptr, ptr, ptr, ptr, ptr, ptr, _I64, _INT, ptr],
    "bz_reversi_terminal": [ptr, ptr, ptr, ptr, ptr, ptr, _I64, _INT, ptr],
    "bz_reversi_step_first_legal": [ptr, ptr, ptr, ptr, ptr, ptr, _I64, _INT, ptr],
    "bz_reversi_planes": [ptr, ptr, ptr, _I64, ptr],
    "bz_ttt_legal_mask": [ptr, ptr, ptr, _I64, ptr],
    "bz_ttt_apply": [ptr, ptr, ptr, ptr, ptr, ptr, ptr, _I64, ptr],
    "bz_ttt_terminal": [ptr, ptr, ptr, ptr, _I64, ptr],
    "bz_mcts_reset": [_PP, ptr, ptr, ptr],
    "bz_mcts_select": [_PP, ptr],
    "bz_mcts_gather": [_PP, ptr],
    "bz_mcts_expand_backup": [_PP, ptr, ptr, ptr],
    "bz_mcts_step": [_PP, ptr, ptr, ptr],
    "bz_mcts_search_fused": [_PP, ptr, ptr, _INT, ptr],
    "bz_mcts_search_fused_entrants": [_PP, ptr, ptr, _INT, ptr, ptr],
    "bz_mcts_root_policy": [_PP, ptr, ptr, ptr, ptr],
    "bz_mcts_root_edges": [_PP, ptr, ptr, ptr, ptr],
    "bz_mcts_best_action": [_PP, ptr, ptr],
    "bz_mcts_root_noise": [_PP, ptr, _F, ptr],
    "bz_mcts_reroot": [_PP, ptr, ptr, ptr, ptr, _INT, ptr, ptr],
    "bz_hash_eval": [ptr, ptr, _U64, _INT, ptr, ptr, _I64, ptr],
    "bz_selfplay_init": [_SP, _I64, ptr],
    "bz_selfplay_advance": [_SP, _PP, ptr, ptr],
    "bz_match_init": [_MP, ptr],
    "bz_match_advance": [_MP, _PP, ptr],
    "bz_tournament_layout": [_TP, ptr],
    "bz_tournament_minimax": [_TP, ptr, ptr, ptr, ptr, ptr],
    "bz_tournament_advance": [_TP, _PP, ptr, ptr, ptr],
    "bz_minimax_moves": [ptr, ptr, ptr, ptr, _U64, _I64, _INT, ptr, ptr, ptr, ptr, ptr],
    "bz_minimax_workspace_bytes": [_I64],
    "bz_endgame_solve": [ptr, ptr, _I64, _INT, ptr, ptr, ptr, ptr, ptr, ptr],
    "bz_endgame_workspace_bytes": [_I64],
    "bz_reversi_symmetry": [ptr, ptr, ptr, ptr, ptr, ptr, ptr, _I64, _INT, ptr],
    "bz_record_hash": [ptr, ptr, ptr, ptr, _I64, ptr],
    "bz_philox_u32": [_U64, ptr, ptr, ptr, _I64, ptr],
    "bz_mlp_forward_pair": [ptr, ptr, ptr, _I64, ptr],
    "bz_mlp_pair_image_bytes": [],
    "bz_mlp_forward_pair2": [ptr, ptr, ptr, _I64, ptr],
    "bz_int32_microbench": [ptr, _INT, _INT, _INT, _INT, C.POINTER(C.c_int64), ptr],
}


class BzError(RuntimeError):
    pass


def lib_path() -> str:
    return _build.LIB


ABI_VERSION = 6  # BZ_ABI_VERSION of include/betazero_b200.h this module's structs and signatures mirror


def load():
    """dlopen the CUDA library, building it first if needed.  Fails loudly."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("BETAZERO_B200_LIB") or _build.LIB  # override: kernel-variant experiments
    if path == _build.LIB and _build.needs_build():
        try:
            _build._nvcc()
        except RuntimeError as e:  # no compiler: a box that received a prebuilt .so may still run it
            if not os.path.exists(path):
                raise BzError(f"libbetazero_b200.so is missing and could not be built ({e}); "
                              "there is no CPU fallback") from e
            import warnings

            warnings.warn("libbetazero_b200.so does not match the sources' hash and nvcc is not available to rebuild "
                          "it: loading the existing library as is", RuntimeWarning)
        else:
            _build.build()  # a compile error in edited sources propagates: never run a stale library silently
    lib = C.CDLL(path)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library lacks a declared symbol
        fn.argtypes = argtypes
        fn.restype = C.c_char_p if name == "bz_error_string" else (C.c_int64 if name.endswith("_bytes") else C.c_int)
    if lib.bz_abi_version() != ABI_VERSION:  # a stale prebuilt library: the struct layouts would not match
        raise BzError(f"libbetazero_b200.so has ABI version {lib.bz_abi_version()}, this package needs {ABI_VERSION}; rebuild it")
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().bz_error_string(rc)
        raise BzError(f"{what or 'bz call'} failed: {msg.decode() if msg else rc} (code {rc})")


def stream_ptr():
    import torch

    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def dptr(t):
    """device pointer of a CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise BzError("expected a CUDA tensor: the engine has no CPU path")
    if not t.is_contiguous():
        raise BzError("expected a contiguous tensor")
    return C.c_void_p(t.data_ptr())


_pdl_state = None  # last value given to bz_set_pdl (None: not set yet, the library default is off)


def set_pdl(enable: bool) -> bool:
    """Process-wide switch for programmatic dependent launch between the tree step kernel and the
    fused MLP kernel (bz_set_pdl).  Returns the previous setting.  The launch attribute is only safe
    when a step kernel never directly follows another step kernel in the stream (its prologue reads
    tree state before it waits for the previous grid), so ``BatchedMCTS`` sets it before every launch
    from its evaluator's ``pdl`` attribute; the cached value makes the repeated call free."""
    global _pdl_state
    enable = bool(enable)
    if _pdl_state is enable:
        return enable
    prev = bool(load().bz_set_pdl(1 if enable else 0))
    _pdl_state = enable
    return prev
