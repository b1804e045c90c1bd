"""ctypes binding of libxq_b200.so (the C ABI declared in include/xq.h).

There is no CPU implementation behind this module: if the CUDA library is missing the import
fails loudly, and every compute call fails with XQ_ERR_CUDA when no B200 is visible.
"""
import ctypes as C
import os

import numpy as np

from . import build as _build

ENV_DTYPE = np.dtype([("sq", "<u4", (12,)), ("move_count", "<u2"), ("player", "u1"), ("flags", "u1"),
                      ("red_score", "<i4"), ("black_score", "<i4"), ("ctr", "<u4")])
TRACE_DTYPE = np.dtype([("action", "<u2"), ("n_legal", "u1"), ("flags", "u1"), ("reward", "<i4")])
STATS_DTYPE = np.dtype([("steps", "<u8"), ("games", "<u8"), ("red_wins", "<u8"), ("black_wins", "<u8"),
                        ("cap_games", "<u8"), ("captures", "<u8"), ("reward_sum", "<i8"), ("legal_sum", "<u8")])
TRANSITION_DTYPE = np.dtype([("s", "<u4", (12,)), ("s2", "<u4", (12,)), ("action", "<u2"), ("mover", "u1"), ("done", "u1"),
                             ("reward", "<i4"), ("reserved", "<u4", (6,))])
assert TRANSITION_DTYPE.itemsize == 128
MAX_ACTIONS = 128
STATE_SIZE = 1260
POLICY_ACTIONS = 8100     # policy index = from * 90 + to (include/xq.h: XQ_POLICY_ACTIONS)
MASK_WORDS = 254          # uint32 words of a packed legal-action mask
DTYPE_F32, DTYPE_BF16, DTYPE_U8 = 0, 1, 2
VIEW_ABSOLUTE, VIEW_SIDE_TO_MOVE = 0, 1
PICK_GREEDY, PICK_SAMPLE, PICK_GIVEN = 0, 1, 2
SEARCH_MAX_EDGES = 128    # edge slots per search-tree node (include/xq.h: XQ_SEARCH_MAX_EDGES)
SEARCH_ADVANCE_MAX_SIMULATIONS = 65536    # largest max_simulations xq_search_advance takes (include/xq.h)
SEARCH_MAX_LEAVES = 32    # largest max_leaves of a search, leaves of one selection (include/xq.h: XQ_SEARCH_MAX_LEAVES)
SEARCH_NODE_DTYPE = np.dtype([("rec", ENV_DTYPE), ("parent", "<i4"), ("visits", "<i4"), ("reward", "<i4"), ("depth", "<i4"),
                              ("parent_edge", "u1"), ("n_edges", "u1"), ("expanded", "u1"), ("status", "u1"), ("winner", "u1"),
                              ("reserved", "u1", (3,))])
SEARCH_EDGE_DTYPE = np.dtype([("action", "<i4"), ("prior", "<f4"), ("visits", "<i4"), ("value_sum", "<f4"), ("child", "<i4")])
assert SEARCH_NODE_DTYPE.itemsize == 88 and SEARCH_EDGE_DTYPE.itemsize == 20
EXAMPLE_DTYPE = np.dtype([("rec", ENV_DTYPE), ("env", "<u8"), ("game", "<u4"), ("ply", "<u2"), ("n_edges", "u1"), ("reserved0", "u1"),
                          ("z", "<f4"), ("q", "<f4"), ("total_visits", "<u4"), ("reserved1", "<u4"), ("action", "<i2", (128,)),
                          ("visits", "<u4", (128,))])
assert EXAMPLE_DTYPE.itemsize == 864


class XQError(RuntimeError):
    pass


_P = C.c_void_p
_lib = None


def lib():
    """Load (never build implicitly on a GPU box) the native library."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB
    if not os.path.exists(path):
        raise XQError(f"{path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                      "(there is no CPU fallback for the hot path)")
    L = C.CDLL(path)
    L.xq_last_error.restype = C.c_char_p
    L.xq_version.restype = C.c_char_p
    L.xq_launch_count.restype = C.c_uint64
    L.xq_rng.restype = C.c_uint64
    L.xq_rng.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32]
    L.xq_eps_threshold.restype = C.c_uint32
    L.xq_eps_threshold.argtypes = [C.c_double]
    L.xq_device_count.argtypes = [C.POINTER(C.c_int)]
    L.xq_env_create.argtypes = [C.c_int64, C.c_int, C.c_uint64, C.c_uint64, C.POINTER(_P)]
    for f in ("xq_env_destroy", "xq_env_sync"):
        getattr(L, f).argtypes = [_P]
    L.xq_env_count.argtypes = [_P, C.POINTER(C.c_int64)]
    L.xq_env_set_stream.argtypes = [_P, _P]
    L.xq_env_device_boards.argtypes = [_P, C.POINTER(_P)]
    L.xq_env_reset.argtypes = [_P, _P]
    L.xq_env_set_boards.argtypes = [_P, _P, C.c_int64, C.c_int64]
    L.xq_env_get_boards.argtypes = [_P, _P, C.c_int64, C.c_int64]
    L.xq_env_legal_moves.argtypes = [_P, _P, _P]
    L.xq_env_legal_moves_strict.argtypes = [_P, _P, _P]
    L.xq_env_valid_moves.argtypes = [_P, C.c_int, C.c_int, _P, _P]
    L.xq_env_is_valid_move.argtypes = [_P, _P, _P]
    L.xq_env_step.argtypes = [_P, _P, _P, _P, _P, _P, _P, C.c_int]
    L.xq_env_rollout_random.argtypes = [_P, C.c_int, _P, _P]
    L.xq_env_rollout_random_io.argtypes = [_P, _P, C.c_int, _P, _P, _P]
    L.xq_env_rollout_random_io_submit.argtypes = [_P, _P, C.c_int, _P, _P, _P]
    L.xq_env_rollout_random_io_wait.argtypes = [_P]
    L.xq_env_rollout_random_async.argtypes = [_P, C.c_int]
    L.xq_env_rollout_random_traced_async.argtypes = [_P, C.c_int, C.POINTER(_P)]
    L.xq_env_legal_moves_device.argtypes = [_P, C.POINTER(_P), C.POINTER(_P)]
    L.xq_env_pick_random_device.argtypes = [_P, C.POINTER(_P)]
    L.xq_env_step_device.argtypes = [_P, _P, C.c_int] + [C.POINTER(_P)] * 5
    L.xq_env_get_stats.argtypes = [_P, _P, C.c_int]
    L.xq_env_state_onehot.argtypes = [_P, _P]
    L.xq_env_observe_device.argtypes = [_P, _P, C.c_int, C.c_int, _P]
    L.xq_env_legal_mask_device.argtypes = [_P, _P, C.c_int, C.c_int]
    L.xq_env_policy_step_device.argtypes = [_P, _P, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int] + [_P] * 7
    L.xq_search_create.argtypes = [_P, C.c_int, C.POINTER(_P)]
    L.xq_search_create_ex.argtypes = [_P, C.c_int, C.c_int, C.POINTER(_P)]
    L.xq_search_destroy.argtypes = [_P]
    L.xq_search_bytes_per_tree.argtypes = [C.c_int, C.POINTER(C.c_int64)]
    L.xq_search_bytes_per_tree_ex.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_int64)]
    L.xq_search_reset.argtypes = [_P]
    L.xq_search_advance.argtypes = [_P, C.c_int, _P, C.c_float, C.c_int, _P]
    L.xq_search_select_device.argtypes = [_P, C.c_float, C.c_float, _P, _P, _P, _P]
    L.xq_search_select_leaves_device.argtypes = [_P, C.c_int, C.c_float, C.c_float, C.c_float, _P, _P, _P, _P]
    L.xq_search_leaves_device.argtypes = [_P, C.POINTER(_P)]
    L.xq_search_observe_leaves_device.argtypes = [_P, _P, C.c_int, C.c_int, _P]
    L.xq_search_expand_backup_device.argtypes = [_P, _P, C.c_int, C.c_float, C.c_int, _P, _P, C.c_float]
    L.xq_search_root_device.argtypes = [_P, C.c_int, _P, _P, _P]
    L.xq_search_play_device.argtypes = [_P, C.c_float, C.c_int, C.c_int, C.c_int] + [_P] * 6
    L.xq_search_root_noise_device.argtypes = [_P, C.c_float, C.c_float, C.c_uint64, _P, _P]
    L.xq_search_get_tree.argtypes = [_P, C.c_int64, _P, _P, C.POINTER(C.c_int32)]
    L.xq_examples_create.argtypes = [_P, C.c_int64, C.c_int, C.POINTER(_P)]
    L.xq_examples_destroy.argtypes = [_P]
    L.xq_examples_bytes.argtypes = [C.c_int64, C.c_int64, C.c_int, C.POINTER(C.c_int64)]
    L.xq_examples_record_device.argtypes = [_P, _P, _P]
    L.xq_examples_end_games_device.argtypes = [_P, _P, _P]
    L.xq_examples_discard_device.argtypes = [_P, _P]
    L.xq_examples_sample_device.argtypes = [_P, C.c_int64, C.c_uint64, C.c_uint32, C.c_int, _P, C.c_int, _P, _P, _P, _P, _P]
    L.xq_examples_info.argtypes = [_P] + [C.POINTER(C.c_int64)] * 6
    L.xq_examples_get.argtypes = [_P, C.c_int64, C.c_int64, _P]
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise XQError(f"xq error {rc}: {lib().xq_last_error().decode(errors='replace')}")


def ptr(a):
    return None if a is None else a.ctypes.data
