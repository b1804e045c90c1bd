"""cn_chess_ai_b200: B200-native batched Xiangqi environment + DQN trainer (sm_100a only).

Host-side mirror of the C ABI in include/xq.h; the hot path lives in csrc/ as hand-written CUDA.
"""
from ._lib import (ENV_DTYPE, EXAMPLE_DTYPE, MAX_ACTIONS, SEARCH_ADVANCE_MAX_SIMULATIONS, STATE_SIZE, STATS_DTYPE, TRACE_DTYPE,  # noqa: F401
                   TRANSITION_DTYPE, XQError, lib)
from .env import BatchedEnv, BatchedExamples, BatchedSearch, action, examples_bytes, search_bytes_per_tree  # noqa: F401
from .dqn import AS_WRITTEN, CORRECTED, DQN  # noqa: F401
from .replay import ReplayBuffer, act, collect, td_update_replay, td_update_replay_n  # noqa: F401
from .trainer import GAME_EVENT_DTYPE, drain_game_events, enable_game_events, train  # noqa: F401
from .benchmarks import bench_dqn  # noqa: F401


def __getattr__(name):
    """TorchEnv (torch_env.py), TorchSearch (torch_search.py) and TorchExamples (torch_examples.py) are loaded on first use: importing
    the package does not import torch"""
    if name == "TorchEnv":
        from .torch_env import TorchEnv
        return TorchEnv
    if name == "TorchSearch":
        from .torch_search import TorchSearch
        return TorchSearch
    if name == "TorchExamples":
        from .torch_examples import TorchExamples
        return TorchExamples
    raise AttributeError(f"module {__name__!r} has no attribute {name!r}")
