"""ctypes binding of libfpc.so (the C-ABI in include/fpc.h).

There is no CPU fallback: if the library is missing this module raises at import of the symbol
table, and every compute call fails with FPC_ERR_CUDA when no B200 is visible."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# FPC_LIB_PATH loads another build of the library instead, e.g. to compare two builds with bench.py
LIB_PATH = os.environ.get("FPC_LIB_PATH") or os.path.join(_HERE, "libfpc.so")

FPC_MAX_MOVES = 300
FPC_OK, FPC_ERR_ARG, FPC_ERR_CUDA, FPC_ERR_MOVE, FPC_ERR_OVERFLOW = 0, -1, -2, -3, -4
STATUS_RESULT_MASK, STATUS_IN_CHECK, STATUS_CAN_TAKE_KING = 0x3, 0x100, 0x200
STATUS_OVERFLOW, STATUS_FINISHED, STATUS_CHECK = 0x400, 0x800, 0x1000
FLAG_ASYNC_DENSE = 1
FLAG_INCREMENTAL = 2
TREE_ADVANCE_MAX_NODE_CAP = 524288
MAX_LEAVES_PER_GAME = 256
SLOT_EMPTY, SLOT_LEAF, SLOT_COLLISION = 0, 1, 2

_vp, _i, _u64 = C.c_void_p, C.c_int, C.c_uint64

# name -> (restype, argtypes); mirrors include/fpc.h one to one
SIGNATURES = {
    "fpc_last_error": (C.c_char_p, []),
    "fpc_version": (_i, []),
    "fpc_supported": (_i, [_i]),
    "fpc_invalid_area": (_i, [_i]),
    "fpc_record_bytes": (_i, [_i]),
    "fpc_num_action_channels": (_i, [_i]),
    "fpc_action_space_size": (_i, [_i]),
    "fpc_state_space_size": (_i, [_i]),
    "fpc_move_from_flat": (_u64, [_i, _i]),
    "fpc_move_flat_index": (_i, [_i, _u64]),
    "fpc_record_from_fen": (_i, [_i, C.c_char_p, _i, _vp]),
    "fpc_observe": (_i, [_i, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _i, _vp]),
    "fpc_observe_tracked": (_i, [_vp, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _i, _vp]),
    "fpc_dense_track_create": (_vp, [_i, _i]),
    "fpc_dense_track_invalidate": (None, [_vp]),
    "fpc_dense_track_destroy": (None, [_vp]),
    "fpc_shutdown": (_i, []),
    "fpc_join": (_i, [_vp]),
    "fpc_profile_enable": (_i, [_i]),
    "fpc_profile_read": (_i, [_vp, _vp, _vp]),
    "fpc_encode": (_i, [_i, _vp, _i, _vp, _i, _vp, _i, _vp]),
    "fpc_make_moves": (_i, [_i, _vp, _vp, _i, _vp, _vp, _vp]),
    "fpc_make_index": (_i, [_i, _vp, _vp, _i, _vp, _vp, _vp]),
    "fpc_heuristic": (_i, [_i, _vp, _i, _vp, _vp]),
    "fpc_playout_step": (_i, [_i, _vp, _i, _u64, _vp, _vp, _vp, _i, _u64, _vp, _vp, _vp, _vp, _vp, _i, _vp,
                              _vp, _i, _vp]),
    "fpc_playout_step_tracked": (_i, [_vp, _i, _vp, _i, _u64, _vp, _vp, _vp, _i, _u64, _vp, _vp, _vp, _vp, _vp, _i, _vp,
                                      _vp, _i, _vp]),
    "fpc_tree_reset": (_i, [_vp, _vp, _vp]),
    "fpc_tree_advance": (_i, [_vp, _vp, _vp, C.c_int32, C.c_int32, _vp, _vp]),
    "fpc_tree_select": (_i, [_vp, _i, _vp, _i, _vp, _vp]),
    "fpc_tree_expand_backup": (_i, [_vp, _vp, _vp, _vp]),
    "fpc_tree_select_leaves": (_i, [_vp, _vp, _i, _vp, _i, _vp, _vp]),
    "fpc_tree_expand_backup_leaves": (_i, [_vp, _vp, _vp, _vp, _vp]),
    "fpc_tree_root_noise": (_i, [_vp, _u64, _vp, C.c_float, C.c_float, _vp, _vp]),
    "fpc_tree_select_gumbel": (_i, [_vp, _vp, _i, _vp, _i, _vp, _vp]),
    "fpc_tree_gumbel_result": (_i, [_vp, _vp, _vp, _vp, _vp]),
    "fpc_tree_select_gumbel_interior": (_i, [_vp, _vp, _vp, _i, _vp, _i, _vp, _vp]),
    "fpc_tree_select_gumbel_leaves": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _vp, _i, _vp, _vp]),
    "fpc_tree_gumbel_result_leaves": (_i, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "fpc_tree_sample_root": (_i, [_vp, _u64, _vp, C.c_double, _vp, _vp]),
    "fpc_ctx_create": (_vp, [_i, _i, _i]),
    "fpc_ctx_destroy": (None, [_vp]),
    "fpc_ctx_stream": (_vp, [_vp]),
    "fpc_host_observe": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp]),
    "fpc_host_make_moves": (_i, [_vp, _vp, _vp, _i, _vp, _vp]),
    "fpc_host_make_index": (_i, [_vp, _vp, _vp, _i, _vp, _vp]),
    "fpc_host_playout_step": (_i, [_vp, _vp, _i, _u64, _vp, _vp, _vp, _i, _u64, _vp, _vp, _vp, _i, _vp, _i]),
    "fpc_ctx_sync": (_i, [_vp]),
    "fpc_attack_maps": (_i, [_i, _vp, _i, _vp, _vp]),
    "fpc_ctx_set_stream": (_i, [_vp, _vp]),
    "fpc_current_device": (_i, []),
    "fpc_host_alloc": (_vp, [C.c_size_t]),
    "fpc_host_free": (None, [_vp]),
    "fpc_host_expand": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "fpc_host_fetch_moves": (_i, [_vp, _i, _i, _vp]),
    "fpc_host_encode": (_i, [_vp, _vp, _i, _i, _vp]),
    "fpc_host_heuristic": (_i, [_vp, _vp, _i, _vp]),
    "fpc_host_attack_maps": (_i, [_vp, _vp, _i, _vp]),
    "fpc_env_create": (_vp, [_i, _i, _i]),
    "fpc_env_destroy": (None, [_vp]),
    "fpc_env_stream": (_vp, [_vp]),
    "fpc_env_sync": (_i, [_vp]),
    "fpc_env_set_boards": (_i, [_vp, _vp, _i, _i]),
    "fpc_env_get_boards": (_i, [_vp, _vp, _i, _i]),
    "fpc_env_observe": (_i, [_vp, _i, _i]),
    "fpc_env_playout_step": (_i, [_vp, _u64, _vp, _i, _u64, _i, _i]),
    "fpc_env_dlpack": (_vp, [_vp, _i]),
}
ENV_BOARDS, ENV_COUNTS, ENV_STATUS, ENV_MOVES, ENV_FLAT, ENV_PLANES, ENV_MASK, ENV_PLY, ENV_GAME = 1, 2, 4, 8, 16, 32, 64, 128, 256



class TreeDesc(C.Structure):
    """struct fpc_tree (include/fpc.h): the caller-owned device arrays of the batched PUCT trees."""
    _fields_ = ([("R", C.c_int32), ("n_games", C.c_int32), ("node_cap", C.c_int32), ("board_cap", C.c_int32),
                 ("C", C.c_double)] +
                [(name, C.c_void_p) for name in
                 ("parent", "first_child", "n_children", "visits", "move_flat", "board_idx", "value_sum", "prior",
                  "n_nodes", "n_boards", "leaf", "dropped", "error", "boards", "leaf_boards", "leaf_flat",
                  "leaf_counts", "leaf_status", "k")])


class LeafBatchDesc(C.Structure):
    """struct fpc_leaf_batch (include/fpc.h): the leaf-parallel batch's device arrays."""
    _fields_ = ([("L", C.c_int32), ("virtual_loss", C.c_int32)] +
                [(name, C.c_void_p) for name in
                 ("in_flight", "slot_node", "slot_kind", "leaf_boards", "leaf_flat", "leaf_counts", "leaf_status", "k",
                  "priors", "collisions")])


class GumbelDesc(C.Structure):
    """struct fpc_gumbel (include/fpc.h): the Gumbel root search's parameters and per-game device arrays."""
    _fields_ = [("seed", C.c_uint64), ("keys", C.c_void_p), ("max_considered", C.c_int32), ("n_sims", C.c_int32),
                ("scale", C.c_double), ("c_visit", C.c_double), ("c_scale", C.c_double), ("root_value", C.c_void_p)]


_LIB = None


class FpcError(RuntimeError):
    """Raised for every non-zero return code (the reference raises RuntimeError, wrapper.cpp:17-27)."""


def lib() -> C.CDLL:
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -m alphazero_4_player_chess_b200.build` "
                "(there is no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _LIB = L
    return _LIB


def check(rc: int) -> None:
    if rc != FPC_OK:
        raise FpcError(f"fpc error {rc}: {lib().fpc_last_error().decode()}")
