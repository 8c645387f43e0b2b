"""ctypes binding of include/gmz.h.  There is NO fallback: if libgmz.so is missing or a call
fails, this raises -- the product path never routes around the CUDA library."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.environ.get("GMZ_LIB") or os.path.join(HERE, "libgmz.so")   # GMZ_LIB: development override

GMZ_MODE_ALPHAZERO, GMZ_MODE_MUZERO = 0, 1
GMZ_F32, GMZ_F64, GMZ_BF16 = 0, 1, 2
GMZ_ACCUM_F64, GMZ_ACCUM_F32 = 0, 1
GMZ_WINNER_NONE = 2


class GmzConfig(C.Structure):
    _fields_ = [("board_size", C.c_int32), ("n_in_row", C.c_int32), ("num_simulations", C.c_int32),
                ("num_top_actions", C.c_int32), ("mode", C.c_int32), ("num_games", C.c_int32),
                ("max_moves", C.c_int32), ("accum_dtype", C.c_int32),
                ("c_visit", C.c_double), ("c_scale", C.c_double), ("minmax_delta", C.c_double),
                ("discount", C.c_double)]


class GmzTraj(C.Structure):
    _fields_ = [("n_slots", C.c_int32), ("max_moves", C.c_int32), ("fin_cap", C.c_int32), ("reserved", C.c_int32),
                ("policy", C.c_void_p), ("value", C.c_void_p), ("action", C.c_void_p), ("start_board", C.c_void_p),
                ("start_info", C.c_void_p), ("free_slots", C.c_void_p), ("free_top", C.c_void_p),
                ("fin_queue", C.c_void_p), ("fin_count", C.c_void_p)]


class GmzError(RuntimeError):
    pass


_P = C.c_void_p
# name -> (restype, argtypes); every symbol include/gmz.h declares
SIGNATURES = {
    "gmz_version": (C.c_int, []),
    "gmz_last_error": (C.c_char_p, []),
    "gmz_workspace_bytes": (C.c_size_t, [C.POINTER(GmzConfig)]),
    "gmz_create": (C.c_int, [C.POINTER(GmzConfig), _P, C.c_size_t, _P, C.POINTER(_P)]),
    "gmz_destroy": (C.c_int, [_P]),
    "gmz_set_roots": (C.c_int, [_P, _P, _P, _P, _P, _P]),
    "gmz_games_reset": (C.c_int, [_P, _P, _P]),
    "gmz_root_obs": (C.c_int, [_P, _P, C.c_int, _P]),
    "gmz_get_roots": (C.c_int, [_P, _P, _P, _P, _P, _P]),
    "gmz_root_expand": (C.c_int, [_P, _P, _P, C.c_int, _P, _P]),
    "gmz_select": (C.c_int, [_P, _P, C.c_int, _P, _P, _P]),
    "gmz_select_mz": (C.c_int, [_P, _P, _P, _P, _P, _P, _P]),
    "gmz_expand_backup": (C.c_int, [_P, _P, _P, _P, C.c_int, _P]),
    "gmz_finalize": (C.c_int, [_P, _P, _P, _P, _P, _P]),
    "gmz_e0_eval_obs": (C.c_int, [_P, C.c_int, C.c_int, C.c_uint64, C.c_int, _P, _P, _P]),
    "gmz_search_e0": (C.c_int, [_P, _P, C.c_uint64, C.c_int, _P, _P, _P]),
    "gmz_fill_gumbel": (C.c_int, [_P, C.c_size_t, C.c_uint64, C.c_uint64, _P]),
    "gmz_game_step": (C.c_int, [_P, _P, _P, _P]),
    "gmz_traj_init": (C.c_int, [_P, C.POINTER(GmzTraj), _P]),
    "gmz_selfplay_e0": (C.c_int, [_P, C.POINTER(GmzTraj), C.c_uint64, C.c_int, C.c_uint64, C.c_int64, C.c_int, _P]),
    "gmz_selfplay_unpark": (C.c_int, [_P, C.POINTER(GmzTraj), _P]),
    "gmz_selfplay_step": (C.c_int, [_P, C.POINTER(GmzTraj), _P, _P, _P, C.c_int, _P, _P]),
    "gmz_play_counters": (C.c_int, [_P, _P, _P]),
    "gmz_select_counters": (C.c_int, [_P, _P, _P]),
    "gmz_hidden_gather": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, C.c_int, _P, _P]),
    "gmz_hidden_scatter": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P]),
    "gmz_move_record_bytes": (C.c_size_t, [C.c_int]),
    "gmz_traj_pack": (C.c_int, [C.POINTER(GmzTraj), C.c_int, _P, C.c_int, _P, _P, C.c_int, _P, _P]),
    "gmz_records_batch": (C.c_int, [_P, C.c_int64, C.c_int, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P, _P, _P, _P]),
    "gmz_records_tactics": (C.c_int, [_P, C.c_int64, C.c_int, C.c_int, _P, _P]),
    "gmz_set_roots_from_records": (C.c_int, [_P, _P, C.c_int64, C.c_int64, C.c_int64, _P]),
    "gmz_records_writeback": (C.c_int, [_P, C.c_int64, C.c_int, C.c_int64, C.c_int64, _P, _P, _P]),
    "gmz_records_retarget": (C.c_int, [_P, C.c_int64, C.c_int, C.c_int64, C.c_int64, _P, C.c_int, _P]),
    "gmz_records_compact": (C.c_int, [_P, C.c_int64, C.c_int, C.c_int64, C.c_int64, _P, _P, _P, _P]),
    "gmz_records_expand": (C.c_int, [_P, _P, C.c_int64, _P, _P, C.c_int64, C.c_int64, C.c_int, _P, C.c_int64, C.c_int64, _P]),
    "gmz_tactics_classify": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P, _P]),
    "gmz_per_update": (C.c_int, [_P, C.c_int64, _P, _P, C.c_int, _P]),
    "gmz_per_add": (C.c_int, [_P, C.c_int64, C.c_int64, _P, C.c_int, _P, _P]),
    "gmz_per_sample": (C.c_int, [_P, C.c_int64, C.c_int64, _P, C.c_int, C.c_double, _P, _P, _P, _P]),
}

_lib = None


def load():
    """Load libgmz.so (built in-tree by __graft_entry__.build()).  Raises if it is absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO):
            raise GmzError(f"{SO} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback)")
        lib = C.CDLL(SO)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)       # AttributeError if a declared symbol is missing
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def check(rc: int, what: str = "gmz"):
    if rc != 0:
        raise GmzError(f"{what} failed: {load().gmz_last_error().decode()}")
