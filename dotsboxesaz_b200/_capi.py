"""ctypes binding of include/dbaz_b200.h.  There is no CPU fallback: if the CUDA library is
missing or no device is present, importing the engine raises."""
import ctypes as C
import os

import numpy as np

from . import _build

MAX_ACTIONS = 128
RESULT_NONE = 2
F32, F16, BF16, I16 = 0, 1, 2, 3
NCHW, NHWC = 0, 1

# host view of the packed 32-byte state (include/dbaz_b200.h: dbaz_state)
STATE_DTYPE = np.dtype([("edges", "<u8", (2,)), ("btc2", "<i2", (2,)), ("to_play", "u1"), ("just_played", "i1"),
                        ("flags", "u1"), ("depth", "u1"), ("parent", "<i4"), ("parent_action", "<i2"), ("result", "<i2")])
assert STATE_DTYPE.itemsize == 32


class Config(C.Structure):
    _fields_ = [("abi_version", C.c_int32), ("device", C.c_int32), ("board_l", C.c_int32), ("board_c", C.c_int32),
                ("n_games", C.c_int32), ("max_nodes", C.c_int32), ("lut_size", C.c_int32), ("max_pending", C.c_int32),
                ("cpuct", C.c_double), ("cpuct_base", C.c_double)]


class SelfplayBuffers(C.Structure):
    """dbaz_selfplay_buffers (include/dbaz_b200.h): device pointers of the asynchronous self-play loop."""
    _fields_ = [("n_moves", C.c_int32), ("reserved", C.c_int32)] + [(k, C.c_void_p) for k in (
        "inv_temp", "uniforms", "noise", "reads_by_k", "searching", "move_idx", "moves", "h_states", "h_visits", "h_active",
        "h_moves", "h_stats", "h_q", "noise_buf", "reads", "left")]


# every symbol include/dbaz_b200.h declares: name -> (restype, argtypes)
_P, _I64, _U64, _I32, _D = C.c_void_p, C.c_int64, C.c_uint64, C.c_int32, C.c_double
SYMBOLS = {
    "dbaz_abi_version": (C.c_int, []),
    "dbaz_sizeof_state": (C.c_int, []),
    "dbaz_engine_create": (C.c_int, [C.POINTER(Config), C.POINTER(_P)]),
    "dbaz_engine_destroy": (None, [_P]),
    "dbaz_last_error": (C.c_char_p, [_P]),
    "dbaz_engine_info": (C.c_int, [_P, _P]),
    "dbaz_engine_set_cpuct": (C.c_int, [_P, _D, _D]),
    "dbaz_game_init": (C.c_int, [_P, _P, _I64, _U64]),
    "dbaz_game_valid_moves": (C.c_int, [_P, _P, _P, _I64, _U64]),
    "dbaz_game_play": (C.c_int, [_P, _P, _P, _P, _P, _I64, _U64]),
    "dbaz_game_result": (C.c_int, [_P, _P, _P, _I64, _U64]),
    "dbaz_game_features": (C.c_int, [_P, _P, _P, _I32, _I32, _I64, _U64]),
    "dbaz_game_random_rollout": (C.c_int, [_P, _P, _U64, _U64, _P, _P, _I32, _I64, _U64]),
    "dbaz_search_reset_roots": (C.c_int, [_P, _P, _U64]),
    "dbaz_search_begin": (C.c_int, [_P, _P, _I32, _P, _D, _U64]),
    "dbaz_search_step": (C.c_int, [_P, _P, _P, _P, _I32, _I32, _P, _P, _U64]),
    "dbaz_search_loop_build": (C.c_int, [_P, _P, _P, _P, _I32, _I32, C.c_float, C.c_float, C.c_float, C.c_float, _P]),
    "dbaz_search_loop_pick": (C.c_int, [_P, _P, _I32, C.c_float, C.c_float, C.c_float, _I32]),
    "dbaz_search_loop_launch": (C.c_int, [_P, _U64, _U64]),
    "dbaz_search_loop_counts": (C.c_int, [_P, _U64, _P, _U64]),
    "dbaz_search_loop_destroy": (None, [_P, _U64]),
    "dbaz_search_stop": (C.c_int, [_P, _U64]),
    "dbaz_search_root_visits": (C.c_int, [_P, _P, _U64]),
    "dbaz_search_root_children": (C.c_int, [_P, _P, _P, _P, _P, _U64]),
    "dbaz_search_tree_stats": (C.c_int, [_P, _P, _P, _P, _U64]),
    "dbaz_search_root_states": (C.c_int, [_P, _P, _U64]),
    "dbaz_search_node": (C.c_int, [_P, _I32, _I32, _P, _P, _P, _P, _P, _P, _P, _P, _P, _U64]),
    "dbaz_search_tree_busy": (C.c_int, [_P, _P, _U64]),
    "dbaz_search_advance_roots": (C.c_int, [_P, _P, _I32, _U64]),
    "dbaz_selfplay_pick": (C.c_int, [_P, C.POINTER(SelfplayBuffers), _U64]),
    "dbaz_selfplay_restart": (C.c_int, [_P, C.POINTER(SelfplayBuffers), _I32, _U64]),
    "dbaz_selfplay_adjudicate": (C.c_int, [_P, C.POINTER(SelfplayBuffers), _P, _I32, _I32, _U64]),
    "dbaz_selfplay_exact_endgame": (C.c_int, [_P, C.POINTER(SelfplayBuffers), _P, _I32, _I32, _I32, _U64]),
    "dbaz_search_status": (C.c_int, [_P, _P, _U64]),
    "dbaz_search_set_mode": (C.c_int, [_P, _I32, _I32]),
    "dbaz_search_set_chain_budget": (C.c_int, [_P, _I32]),
    "dbaz_search_wave_counts": (C.c_int, [_P, _P, _U64]),
    "dbaz_search_set_batch_rows": (C.c_int, [_P, _I32]),
    "dbaz_cache_configure": (C.c_int, [_P, _I32]),
    "dbaz_cache_clear": (C.c_int, [_P, _U64]),
    "dbaz_nn_stem": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _I32, _I32, _I32, _I64, _U64]),
    "dbaz_nn_stem_mma_pack": (C.c_int, [_P, _P, _P, _I32, _U64]),
    "dbaz_nn_stem_mma": (C.c_int, [_P, _P, _P, _P, _I32, _I32, _I64, _U64]),
    "dbaz_nn_heads": (C.c_int, [_P, _P, _I32, _I32, _P, _P, _I64, _U64]),
    "dbaz_nn_heads_mlp": (C.c_int, [_P, _P, _I32, _I32, _I32, _P, _P, _P, _I64, _U64]),
    "dbaz_nn_tower_geometry": (C.c_int, [_P, _P]),
    "dbaz_nn_stem_mma_tiles": (C.c_int, [_P, _P, _P, _P, _I64, _U64]),
    "dbaz_nn_tower_planarize": (C.c_int, [_P, _P, _P, _I64, _U64]),
    "dbaz_nn_tower": (C.c_int, [_P, _P, _P, _P, _I32, _I32, _P, _I64, _U64]),
    "dbaz_nn_tower_trace": (C.c_int, [_P, _P]),
    "dbaz_nn_trunk_conv_taps": (C.c_int, [_I32, _I32, _I32, _P]),
    "dbaz_nn_trunk_conv_plan_bytes": (C.c_int64, []),
    "dbaz_nn_trunk_conv_plan": (C.c_int, [_P, _P, _P, _P, _P, _P, _I64, _I32, _I32, _I32, _P]),
    "dbaz_nn_trunk_conv": (C.c_int, [_P, _P, _I64, _U64]),
    "dbaz_fake_nn": (C.c_int, [_P, _P, _P, _P, _I32, _I64, _U64]),
    "dbaz_solver_solve": (C.c_int, [_P, _P, _I64, _U64]),
    "dbaz_solver_moves": (C.c_int, [_P, _P, _P, _P, _P, _I64, _U64]),
    "dbaz_solver_eval": (C.c_int, [_P, _P, _P, _P, _P, _I32, _I64, _U64]),
    "dbaz_endgame_moves": (C.c_int, [_P, _P, _P, _P, _I32, _I64, _U64]),
    "dbaz_endgame_eval": (C.c_int, [_P, _P, _P, _P, _I32, _I32, _I32, _I64, _U64]),
    "dbaz_endgame_deep_moves": (C.c_int, [_P, _P, _I64, _I32, _P, _I64, _P, _P, _U64]),
}
TRUNK_MAX_POS = 64  # input positions of dbaz_nn_trunk_conv (the largest board the engine plays)
ENDGAME_DEEP_GEOM_BYTES = 512  # workspace bytes of one position's geometry in dbaz_endgame_deep_moves, beside its 2^f table

_lib = None


def load():
    """dlopen the in-tree CUDA library (building it first when sources are newer)."""
    global _lib
    if _lib is None:
        path = _build.LIB
        if not os.path.exists(path) or os.environ.get("DBAZ_REBUILD"):
            path = _build.build()
        lib = C.CDLL(path)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)  # AttributeError if the library does not export the symbol
            fn.restype = res
            fn.argtypes = args
        if lib.dbaz_abi_version() != 1 or lib.dbaz_sizeof_state() != STATE_DTYPE.itemsize:
            raise RuntimeError("libdbaz_b200.so ABI mismatch")
        _lib = lib
    return _lib
