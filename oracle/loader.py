"""ctypes bindings for the oracle libraries (TEST INFRASTRUCTURE ONLY).

* ``oracle()``  -> oracle/_build/libxq_oracle.so, the plain-C restatement (oracle/xq_oracle.c)
* ``ref()``     -> oracle/_ref/libxq_ref.so, the reference's own sources compiled unmodified
                   (None when it has not been built and XQ_REFERENCE_SRC names no checkout of the
                   reference project to build it from; the tests that need it skip then)
"""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF_SRC = os.environ.get("XQ_REFERENCE_SRC", "")

ENV_DTYPE = np.dtype([("sq", "<u4", (12,)), ("move_count", "<u2"), ("player", "u1"), ("flags", "u1"),
                      ("red_score", "<i4"), ("black_score", "<i4"), ("ctr", "<u4")])
TRACE_DTYPE = np.dtype([("action", "<u2"), ("n_legal", "u1"), ("flags", "u1"), ("reward", "<i4")])
STATS_DTYPE = np.dtype([("steps", "<u8"), ("games", "<u8"), ("red_wins", "<u8"), ("black_wins", "<u8"),
                        ("cap_games", "<u8"), ("captures", "<u8"), ("reward_sum", "<i8"), ("legal_sum", "<u8")])
assert ENV_DTYPE.itemsize == 64 and TRACE_DTYPE.itemsize == 8 and STATS_DTYPE.itemsize == 64


def build(force=False):
    """Compile the C restatement, and the verbatim reference when XQ_REFERENCE_SRC names a checkout of it."""
    targets = ["oracle"]
    if os.path.isdir(REF_SRC):
        targets += ["ref", "REF=" + os.path.abspath(REF_SRC)]
    args = ["make", "-C", HERE] + (["-B"] if force else []) + targets
    subprocess.run(args, check=True, stdout=subprocess.DEVNULL)
    if os.path.isdir(REF_SRC) and os.path.exists("/usr/local/cuda/bin/nvcc"):
        # the reference's own CUDA network (src/dqn.cu unmodified, sm_100a): golden generation on a B200 and bench.py's reference_train leg;
        # optional -- without it that leg times the CPU definition of the network
        subprocess.run(["make", "-C", HERE] + (["-B"] if force else []) + ["refcuda", "REF=" + os.path.abspath(REF_SRC)], check=False, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)


_P = C.c_void_p
_u8p = np.ctypeslib.ndpointer(np.uint8, flags="C")
_u16p = np.ctypeslib.ndpointer(np.uint16, flags="C")
_i32p = np.ctypeslib.ndpointer(np.int32, flags="C")
_f64p = np.ctypeslib.ndpointer(np.float64, flags="C")

_oracle = None
_ref = None


def oracle():
    global _oracle
    if _oracle is None:
        path = os.path.join(HERE, "_build", "libxq_oracle.so")
        if not os.path.exists(path):
            build()
        L = C.CDLL(path)
        L.xqo_rng.restype = C.c_uint64
        L.xqo_rng.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32]
        L.xqo_bench_rollout_random.restype = C.c_double
        L.xqo_bench_rollout_random.argtypes = [C.c_int, C.c_long, C.c_int, C.c_uint64, C.POINTER(C.c_long)]
        L.xqo_rollout_random.argtypes = [_P, C.c_long, C.c_uint64, C.c_uint64, C.c_int, _P, _P]
        L.xqo_batch_all_actions.argtypes = [_P, C.c_long, _u8p, _u16p]
        L.xqo_batch_all_actions_strict.argtypes = [_P, C.c_long, _u8p, _u16p]
        L.xqo_batch_step.argtypes = [_P, C.c_long, _u16p, _i32p, _u8p, _u8p, _u8p, _u8p]
        L.xqo_eps_threshold.restype = C.c_uint32
        L.xqo_eps_threshold.argtypes = [C.c_double]
        L.xqo_select_action.argtypes = [_f64p, _u16p, C.c_int, C.c_uint32, C.c_uint32, C.c_double]
        L.xqo_nn_forward.argtypes = [_i32p, C.c_int, _f64p, _f64p, _f64p, _f64p]
        L.xqo_nn_backprop.argtypes = [_i32p, C.c_int, _f64p, _f64p, _f64p, _f64p, C.c_double, C.c_int]
        L.xqo_nn_grad.argtypes = [_i32p, C.c_int, _f64p, _f64p, _f64p, _f64p, C.c_int, _f64p, _f64p]
        L.xqo_td_target.argtypes = [_f64p, _f64p, C.c_int, C.c_int, C.c_double, C.c_int, C.c_double, _f64p]
        L.xqo_td_batch_grad.argtypes = [_i32p, C.c_int, _f64p, _f64p, _f64p, _f64p, _f64p, _f64p, _i32p, _i32p, _u8p, C.c_double, C.c_int, C.c_long,
                                        C.c_int, _f64p, _f64p, C.POINTER(C.c_double)]
        L.xqo_state.argtypes = [_P, _f64p]
        for f in ("xqo_is_valid_move", "xqo_move"):
            getattr(L, f).argtypes = [_P, C.c_int, C.c_int, C.c_int, C.c_int]
        L.xqo_evaluate.argtypes = [_P, C.c_int, C.c_int]
        L.xqo_evaluate_int.argtypes = [_P, C.c_int, C.c_int]
        L.xqo_valid_moves.argtypes = [_P, C.c_int, C.c_int, _u8p]
        L.xqo_all_actions.argtypes = [_P, C.c_int, _u16p]
        for f in ("xqo_reset", "xqo_game_over", "xqo_winner"):
            getattr(L, f).argtypes = [_P]
        _oracle = L
    return _oracle


def ref():
    global _ref
    if _ref is None:
        path = os.path.join(HERE, "_ref", "libxq_ref.so")
        if not os.path.exists(path):
            if not os.path.isdir(REF_SRC):
                return None
            build()
        L = C.CDLL(path)
        L.ref_env_new.restype = _P
        L.ref_dqn_new.restype = _P
        L.ref_last_error.restype = C.c_char_p
        L.ref_bench_rollout_random.restype = C.c_double
        L.ref_bench_rollout_random.argtypes = [C.c_int, C.c_long, C.c_uint64, C.POINTER(C.c_long)]
        L.ref_env_rollout_random.restype = C.c_long
        L.ref_rand_consumed.restype = C.c_long
        L.ref_dqn_num_weights.restype = C.c_long
        L.ref_dqn_num_biases.restype = C.c_long
        for name in ("ref_env_free", "ref_env_reset", "ref_env_game_over", "ref_env_winner", "ref_dqn_free",
                     "ref_dqn_num_weights", "ref_dqn_num_biases", "ref_dqn_update_target"):
            getattr(L, name).argtypes = [_P]
        L.ref_env_get.argtypes = [_P, _u8p, _i32p]
        L.ref_env_set.argtypes = [_P, _u8p, _i32p]
        L.ref_env_is_valid_move.argtypes = [_P, C.c_int, C.c_int, C.c_int, C.c_int]
        L.ref_env_valid_moves.argtypes = [_P, C.c_int, C.c_int, _i32p]
        L.ref_env_all_actions.argtypes = [_P, C.c_int, _i32p]
        L.ref_env_all_actions_strict.argtypes = [_P, C.c_int, _i32p]
        L.ref_env_move.argtypes = [_P, C.c_int, C.c_int]
        L.ref_env_evaluate.argtypes = [_P, C.c_int, C.c_int]
        L.ref_env_state.argtypes = [_P, _f64p]
        L.ref_env_rollout_random.argtypes = [_P, np.ctypeslib.ndpointer(np.uint32, flags="C"), C.c_long, _P, _P]
        L.ref_rand_load.argtypes = [_i32p, C.c_long]
        L.ref_dqn_new.argtypes = [_i32p, C.c_int]
        L.ref_dqn_set_params.argtypes = [_P, _f64p, _f64p]
        L.ref_dqn_get_params.argtypes = [_P, _f64p, _f64p]
        L.ref_dqn_forward.argtypes = [_P, _f64p, C.c_int, _f64p, C.c_int]
        L.ref_dqn_backprop.argtypes = [_P, _f64p, C.c_int, _f64p, C.c_int, C.c_double]
        L.ref_dqn_select.argtypes = [_P, _f64p, C.c_int, C.c_double, _i32p, C.c_int, _i32p]
        L.ref_dqn_train.argtypes = [_P, _f64p, C.c_int, C.c_int, C.c_double, _f64p, C.c_int]
        L.ref_dqn_save.argtypes = [_P, C.c_char_p]
        L.ref_dqn_load.argtypes = [_P, C.c_char_p]
        L.ref_ai_train.argtypes = [_P, C.c_int, _P, _P, _P, _P]
        L.ref_ai_selfplay.argtypes = [_P, C.c_int, _P, _P, _P, _P]
        L.ref_ai_get_move.argtypes = [_P, C.c_int, _P, _P, _i32p]
        L.ref_ai_log_game.argtypes = [_P, C.c_int, C.c_int, C.c_int, C.c_int]
        L.ref_events_get.argtypes = [_i32p]
        _ref = L
    return _ref


# ---- helpers shared by tests / smoke / bench -------------------------------------------------
def new_envs(n):
    """n records at the standard opening (ChessBoard::reset)."""
    envs = np.zeros(n, dtype=ENV_DTYPE)
    L = oracle()
    one = np.zeros(1, dtype=ENV_DTYPE)
    L.xqo_reset(one.ctypes.data)
    envs[:] = one[0]
    return envs


def codes_of(env):
    """90 square codes of one record."""
    sq = np.asarray(env["sq"], dtype=np.uint32)
    return np.array([(int(sq[s >> 3]) >> ((s & 7) * 4)) & 15 for s in range(90)], dtype=np.uint8)


def pack_codes(codes):
    sq = np.zeros(12, dtype=np.uint32)
    for s in range(90):
        sq[s >> 3] |= np.uint32(int(codes[s]) << ((s & 7) * 4))
    return sq


def rng_draws(seed, env_id, ctr0, n):
    L = oracle()
    return np.array([L.xqo_rng(seed, env_id, ctr0 + i) for i in range(n)], dtype=np.uint64)


def rng_np(seed, env_ids, ctrs):
    """vectorised xq_rng (numpy uint64 wrap-around arithmetic)"""
    with np.errstate(over="ignore"):
        z = (np.uint64(seed) + np.asarray(env_ids, np.uint64) * np.uint64(0x9E3779B97F4A7C15)
             + np.asarray(ctrs, np.uint64) * np.uint64(0xD1B54A32D192ED03))
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))
