"""BatchedEnv: host-side handle of the batched Xiangqi environment (include/xq.h, xq_env_*).

Mirrors, for N boards at once, the board-facing API the reference's training loop uses
(ChessBoard::reset/getValidMoves/movePiece/checkGameOver/getWinner and
ChessAI::getAllValidActions/evaluateBoard/getStateRepresentation).
"""
import ctypes as C

import numpy as np

from ._lib import (ENV_DTYPE, EXAMPLE_DTYPE, MAX_ACTIONS, SEARCH_EDGE_DTYPE, SEARCH_MAX_EDGES, SEARCH_NODE_DTYPE, STATE_SIZE, STATS_DTYPE, TRACE_DTYPE,
                   check, lib, ptr)


def action(from_sq, to_sq):
    return (from_sq << 7) | to_sq


class BatchedEnv:
    def __init__(self, n_envs, device=0, seed=0, env_id0=0):
        self._L = lib()
        self._h = C.c_void_p()
        check(self._L.xq_env_create(n_envs, device, seed, env_id0, C.byref(self._h)))
        self.n = int(n_envs)
        self.device = device

    def close(self):
        if self._h:
            self._L.xq_env_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        return self._h

    def set_stream(self, cuda_stream):
        check(self._L.xq_env_set_stream(self._h, C.c_void_p(cuda_stream)))

    def sync(self):
        check(self._L.xq_env_sync(self._h))

    def device_boards_ptr(self):
        p = C.c_void_p()
        check(self._L.xq_env_device_boards(self._h, C.byref(p)))
        return p.value

    def reset(self, mask=None):
        m = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        check(self._L.xq_env_reset(self._h, ptr(m)))

    def set_boards(self, recs, first=0):
        recs = np.ascontiguousarray(recs, dtype=ENV_DTYPE)
        check(self._L.xq_env_set_boards(self._h, ptr(recs), first, len(recs)))

    def get_boards(self, first=0, n=None, out=None):
        n = self.n - first if n is None else n
        out = np.empty(n, dtype=ENV_DTYPE) if out is None else out
        check(self._L.xq_env_get_boards(self._h, ptr(out), first, n))
        return out

    def legal_moves(self, strict=False):
        """reference-ordered action lists; strict=True (opt-in, not the reference's rules) drops self-check and flying-general moves"""
        counts = np.empty(self.n, dtype=np.uint8)
        actions = np.empty((self.n, MAX_ACTIONS), dtype=np.uint16)
        check((self._L.xq_env_legal_moves_strict if strict else self._L.xq_env_legal_moves)(self._h, ptr(counts), ptr(actions)))
        return counts, actions

    def valid_moves(self, row, col):
        counts = np.empty(self.n, dtype=np.uint8)
        to = np.empty((self.n, 20), dtype=np.uint8)
        check(self._L.xq_env_valid_moves(self._h, row, col, ptr(counts), ptr(to)))
        return counts, to

    def is_valid_move(self, moves):
        moves = np.ascontiguousarray(moves, dtype=np.int32).reshape(self.n, 4)
        valid = np.empty(self.n, dtype=np.uint8)
        check(self._L.xq_env_is_valid_move(self._h, ptr(moves), ptr(valid)))
        return valid

    def step(self, actions, auto_reset=False):
        actions = np.ascontiguousarray(actions, dtype=np.uint16)
        assert actions.shape == (self.n,)
        reward = np.empty(self.n, dtype=np.int32)
        done, winner, captured, valid = (np.empty(self.n, dtype=np.uint8) for _ in range(4))
        check(self._L.xq_env_step(self._h, ptr(actions), ptr(reward), ptr(done), ptr(winner), ptr(captured), ptr(valid),
                                  1 if auto_reset else 0))
        return reward, done, winner, captured, valid

    def rollout_random(self, n_plies, trace=False):
        tr = np.empty((n_plies, self.n), dtype=TRACE_DTYPE) if trace else None
        stats = np.zeros(1, dtype=STATS_DTYPE)
        check(self._L.xq_env_rollout_random(self._h, n_plies, ptr(tr), ptr(stats)))
        return stats[0], tr

    def rollout_random_io(self, boards_in, n_plies, boards_out, trace=False):
        """host boards in -> n_plies of random-policy self-play -> host boards out, one C-ABI call (one synchronisation)"""
        assert boards_in is None or boards_in.shape == (self.n,)
        assert boards_out is None or boards_out.shape == (self.n,)
        tr = np.empty((n_plies, self.n), dtype=TRACE_DTYPE) if trace else None
        stats = np.zeros(1, dtype=STATS_DTYPE)
        check(self._L.xq_env_rollout_random_io(self._h, ptr(boards_in), n_plies, ptr(boards_out), ptr(tr), ptr(stats)))
        return stats[0], tr

    def rollout_random_io_submit(self, boards_in, n_plies, boards_out, stats_out=None, trace_out=None):
        """first half of rollout_random_io: enqueue and return; the buffers (pinned for the overlap to be real) belong to the library until
        rollout_random_io_wait()"""
        check(self._L.xq_env_rollout_random_io_submit(self._h, ptr(boards_in), n_plies, ptr(boards_out), ptr(trace_out), ptr(stats_out)))

    def rollout_random_io_wait(self):
        check(self._L.xq_env_rollout_random_io_wait(self._h))

    def api_ply_device(self, auto_reset=True):
        """one ply of the API-mode path entirely on the device: ordered lists -> random-policy pick -> movePiece / reward / terminal"""
        check(self._L.xq_env_legal_moves_device(self._h, None, None))
        check(self._L.xq_env_pick_random_device(self._h, None))
        check(self._L.xq_env_step_device(self._h, None, 1 if auto_reset else 0, None, None, None, None, None))

    def legal_moves_device(self):
        check(self._L.xq_env_legal_moves_device(self._h, None, None))

    def rollout_random_async(self, n_plies):
        check(self._L.xq_env_rollout_random_async(self._h, n_plies))

    def stats(self, reset=False):
        stats = np.zeros(1, dtype=STATS_DTYPE)
        check(self._L.xq_env_get_stats(self._h, ptr(stats), 1 if reset else 0))
        return stats[0]

    # ---- device-resident interface for external policies: raw device pointers (ints), asynchronous on the handle's stream ----
    def observe_device(self, planes_ptr, dtype, view, aux_ptr):
        """xq_env_observe_device: planes [n][14][10][9] (dtype DTYPE_*), aux int32 [n][4]; either pointer may be None"""
        check(self._L.xq_env_observe_device(self._h, planes_ptr, dtype, view, aux_ptr))

    def legal_mask_device(self, mask_ptr, packed, view):
        """xq_env_legal_mask_device: uint32 [n][254] (packed) or uint8 [n][8100]"""
        check(self._L.xq_env_legal_mask_device(self._h, mask_ptr, 1 if packed else 0, view))

    def policy_step_device(self, scores_ptr, scores_dtype, pick, temperature, view, auto_reset, actions_ptr, logp_ptr=None, reward_ptr=None,
                           done_ptr=None, winner_ptr=None, captured_ptr=None, valid_ptr=None):
        """xq_env_policy_step_device: one ply from a policy's scores (PICK_GREEDY / PICK_SAMPLE) or given policy indices (PICK_GIVEN)"""
        check(self._L.xq_env_policy_step_device(self._h, scores_ptr, scores_dtype, pick, float(temperature), view, 1 if auto_reset else 0,
                                                actions_ptr, logp_ptr, reward_ptr, done_ptr, winner_ptr, captured_ptr, valid_ptr))

    def legal_actions_device(self, actions_ptr, counts_ptr, view):
        """xq_env_legal_actions_device: int32 [n][128] policy indices of each env's legal actions in list order (-1 past the count),
        counts uint8 [n] or None"""
        check(self._L.xq_env_legal_actions_device(self._h, view, actions_ptr, counts_ptr))

    def policy_step_compact_device(self, scores_ptr, scores_dtype, pick, temperature, view, auto_reset, actions_ptr, logp_ptr=None,
                                   reward_ptr=None, done_ptr=None, winner_ptr=None, captured_ptr=None, valid_ptr=None):
        """xq_env_policy_step_compact_device: policy_step_device with compact scores [n][128] (entry k = list entry k)"""
        check(self._L.xq_env_policy_step_compact_device(self._h, scores_ptr, scores_dtype, pick, float(temperature), view,
                                                        1 if auto_reset else 0, actions_ptr, logp_ptr, reward_ptr, done_ptr, winner_ptr,
                                                        captured_ptr, valid_ptr))

    def state_onehot(self):
        out = np.empty((self.n, STATE_SIZE), dtype=np.float64)
        check(self._L.xq_env_state_onehot(self._h, ptr(out)))
        return out


def search_bytes_per_tree(max_simulations, max_leaves=1):
    """device memory one tree of a BatchedSearch with this capacity (and up to max_leaves leaves per selection) takes"""
    b = C.c_int64()
    check(lib().xq_search_bytes_per_tree_ex(max_simulations, max_leaves, C.byref(b)))
    return b.value


class BatchedSearch:
    """xq_search_*: one PUCT tree per env of `env` (a BatchedEnv), capacity max_simulations simulations per reset, up to max_leaves
    leaves per tree in one selection.  Raw device pointers (ints), asynchronous on the env's stream; close() before the env is closed."""

    def __init__(self, env, max_simulations, max_leaves=1):
        self._L = lib()
        self._h = C.c_void_p()
        check(self._L.xq_search_create_ex(env.handle, max_simulations, max_leaves, C.byref(self._h)))
        self.env = env
        self.n = env.n
        self.max_simulations = int(max_simulations)
        self.max_leaves = int(max_leaves)

    def close(self):
        if self._h:
            self._L.xq_search_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reset(self):
        check(self._L.xq_search_reset(self._h))

    def advance_device(self, min_free, noise_ptr=None, noise_eps=0.0, view=1, kept_ptr=None):
        """xq_search_advance: re-root every tree at its env's current board (keep the played child's subtree, else rebuild the tree);
        min_free more simulations are allowed afterwards.  kept int32 [n]: nodes carried over, 0 for a rebuilt tree"""
        check(self._L.xq_search_advance(self._h, int(min_free), noise_ptr, float(noise_eps), view, kept_ptr))

    def select_device(self, c_puct, fpu, status_ptr=None, winner_ptr=None, reward_ptr=None, depth_ptr=None):
        check(self._L.xq_search_select_device(self._h, float(c_puct), float(fpu), status_ptr, winner_ptr, reward_ptr, depth_ptr))

    def select_leaves_device(self, leaves, c_puct, fpu, virtual_loss, status_ptr=None, winner_ptr=None, reward_ptr=None, depth_ptr=None):
        """xq_search_select_leaves_device: `leaves` leaves per tree with virtual loss; outputs [n][leaves]"""
        check(self._L.xq_search_select_leaves_device(self._h, int(leaves), float(c_puct), float(fpu), float(virtual_loss), status_ptr,
                                                     winner_ptr, reward_ptr, depth_ptr))

    def leaves_device(self):
        """device address of the [n * L] leaf records of the last selection of L leaves"""
        p = C.c_void_p()
        check(self._L.xq_search_leaves_device(self._h, C.byref(p)))
        return p.value

    def observe_leaves_device(self, planes_ptr, dtype, view, aux_ptr):
        check(self._L.xq_search_observe_leaves_device(self._h, planes_ptr, dtype, view, aux_ptr))

    def expand_backup_device(self, scores_ptr, scores_dtype, temperature, view, values_ptr, noise_ptr=None, noise_eps=0.0):
        check(self._L.xq_search_expand_backup_device(self._h, scores_ptr, scores_dtype, float(temperature), view, values_ptr, noise_ptr,
                                                     float(noise_eps)))

    def leaf_actions_device(self, actions_ptr, counts_ptr, view):
        """xq_search_leaf_actions_device: the compact lists int32 [n * L][128] (and counts uint8 [n * L] or None) of the leaf records"""
        check(self._L.xq_search_leaf_actions_device(self._h, view, actions_ptr, counts_ptr))

    def expand_backup_compact_device(self, scores_ptr, scores_dtype, temperature, values_ptr):
        """xq_search_expand_backup_compact_device: expand_backup_device with compact scores [n * L][128] (entry k = edge k)"""
        check(self._L.xq_search_expand_backup_compact_device(self._h, scores_ptr, scores_dtype, float(temperature), values_ptr))

    def root_device(self, view, visits_ptr, q_ptr, best_ptr):
        check(self._L.xq_search_root_device(self._h, view, visits_ptr, q_ptr, best_ptr))

    def play_device(self, temperature, sample_plies, view, auto_reset, actions_ptr=None, reward_ptr=None, done_ptr=None, winner_ptr=None,
                    captured_ptr=None, valid_ptr=None):
        """xq_search_play_device: one move per tree from its root's visit counts (greedy, or sampled with N^(1/temperature) for the first
        sample_plies plies), played on the env"""
        check(self._L.xq_search_play_device(self._h, float(temperature), int(sample_plies), view, 1 if auto_reset else 0, actions_ptr, reward_ptr,
                                            done_ptr, winner_ptr, captured_ptr, valid_ptr))

    def root_noise_device(self, alpha, eps, seed, mask_ptr=None, noise_out_ptr=None):
        """xq_search_root_noise_device: Dirichlet(alpha) noise drawn over each expanded root's edges and mixed into its priors; mask u8 [n]
        or None, noise_out f32 [n][128] (list order) or None"""
        check(self._L.xq_search_root_noise_device(self._h, float(alpha), float(eps), int(seed), mask_ptr, noise_out_ptr))

    def get_tree(self, tree):
        """synchronous read-back of one tree: (nodes SEARCH_NODE_DTYPE [n_nodes], edges SEARCH_EDGE_DTYPE [n_nodes][128])"""
        cap = self.max_simulations + 1
        nodes = np.zeros(cap, SEARCH_NODE_DTYPE)
        edges = np.zeros((cap, SEARCH_MAX_EDGES), SEARCH_EDGE_DTYPE)
        cnt = C.c_int32()
        check(self._L.xq_search_get_tree(self._h, int(tree), ptr(nodes), ptr(edges), C.byref(cnt)))
        return nodes[:cnt.value].copy(), edges[:cnt.value].copy()


def gumbel_bytes(n_trees, max_simulations):
    """device memory a BatchedGumbel on a search of n_trees trees allocates"""
    b = C.c_int64()
    check(lib().xq_gumbel_bytes(int(n_trees), int(max_simulations), C.byref(b)))
    return b.value


class BatchedGumbel:
    """xq_gumbel_*: the Gumbel root-search state of `search` (a BatchedSearch): Gumbel-top-k sampled root actions, Sequential Halving
    over them, and the completed-Q improved policy.  Raw device pointers (ints), asynchronous on the env's stream; close() before the
    search is closed."""

    def __init__(self, search, max_considered=16):
        self._L = lib()
        self._h = C.c_void_p()
        check(self._L.xq_gumbel_create(search._h, int(max_considered), C.byref(self._h)))
        self.search = search
        self.n = search.n
        self.max_considered = int(max_considered)

    def close(self):
        if self._h:
            self._L.xq_gumbel_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def begin_device(self, scores_ptr, scores_dtype, temperature, view, values_ptr, n_simulations, seed, c_visit=50.0, c_scale=0.1):
        """xq_gumbel_begin_device: expand the unexpanded roots from scores [n][8100], then draw the Gumbels, the considered sets, N0 and
        the root values (f32 [n]) of this move's n_simulations"""
        check(self._L.xq_gumbel_begin_device(self._h, scores_ptr, scores_dtype, float(temperature), view, values_ptr, int(n_simulations),
                                             int(seed), float(c_visit), float(c_scale)))

    def begin_compact_device(self, scores_ptr, scores_dtype, temperature, values_ptr, n_simulations, seed, c_visit=50.0, c_scale=0.1):
        """xq_gumbel_begin_compact_device: begin_device with compact root scores [n][128] (entry k = root edge k)"""
        check(self._L.xq_gumbel_begin_compact_device(self._h, scores_ptr, scores_dtype, float(temperature), values_ptr, int(n_simulations),
                                                     int(seed), float(c_visit), float(c_scale)))

    def select_device(self, leaves, c_puct, fpu, virtual_loss, status_ptr=None, winner_ptr=None, reward_ptr=None, depth_ptr=None):
        """xq_gumbel_select_device: xq_search_select_leaves_device with the Gumbel root rule; outputs [n][leaves]"""
        check(self._L.xq_gumbel_select_device(self._h, int(leaves), float(c_puct), float(fpu), float(virtual_loss), status_ptr, winner_ptr,
                                              reward_ptr, depth_ptr))

    def root_device(self, view, policy_ptr=None, action_ptr=None):
        """xq_gumbel_root_device: the improved policy f32 [n][8100] and the action to play int64 [n] (-1 none)"""
        check(self._L.xq_gumbel_root_device(self._h, view, policy_ptr, action_ptr))

    def play_device(self, view, auto_reset, actions_ptr=None, reward_ptr=None, done_ptr=None, winner_ptr=None, captured_ptr=None, valid_ptr=None):
        """xq_gumbel_play_device: the action of root_device played on the env"""
        check(self._L.xq_gumbel_play_device(self._h, view, 1 if auto_reset else 0, actions_ptr, reward_ptr, done_ptr, winner_ptr, captured_ptr,
                                            valid_ptr))

    def get(self, tree):
        """synchronous read-back of one tree's state: dict of gumbel, logit (f32 [128]), n0 (int32 [128]), considered (bool [128]),
        root_value (float) and m (int)"""
        g, lg = np.zeros(SEARCH_MAX_EDGES, np.float32), np.zeros(SEARCH_MAX_EDGES, np.float32)
        n0 = np.zeros(SEARCH_MAX_EDGES, np.int32)
        cons = np.zeros(4, np.uint32)
        v, m = C.c_float(), C.c_int32()
        check(self._L.xq_gumbel_get(self._h, int(tree), ptr(g), ptr(lg), ptr(n0), ptr(cons), C.byref(v), C.byref(m)))
        bits = ((cons[:, None] >> np.arange(32, dtype=np.uint32)[None, :]) & 1).reshape(-1).astype(bool)
        return {"gumbel": g, "logit": lg, "n0": n0, "considered": bits, "root_value": v.value, "m": m.value}


def examples_bytes(n_envs, capacity, max_game_examples):
    """device memory a BatchedExamples of this size allocates (the sampling scratch aside)"""
    b = C.c_int64()
    check(lib().xq_examples_bytes(int(n_envs), int(capacity), int(max_game_examples), C.byref(b)))
    return b.value


class BatchedExamples:
    """xq_examples_*: the self-play example buffer of `env` (a BatchedEnv): per env a staging area of max_game_examples examples for the
    game in progress, a ring of `capacity` committed examples.  Raw device pointers (ints), asynchronous on the env's stream; close()
    before the env is closed."""

    def __init__(self, env, capacity, max_game_examples=256):
        self._L = lib()
        self._h = C.c_void_p()
        check(self._L.xq_examples_create(env.handle, int(capacity), int(max_game_examples), C.byref(self._h)))
        self.env = env
        self.n = env.n
        self.capacity = int(capacity)
        self.max_game_examples = int(max_game_examples)

    def close(self):
        if self._h:
            self._L.xq_examples_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def record_device(self, search, mask_ptr=None):
        """xq_examples_record_device: one example of every root of `search` (a BatchedSearch on the same env), u8 [n] mask or None"""
        check(self._L.xq_examples_record_device(self._h, search._h, mask_ptr))

    def record_gumbel_device(self, gumbel, mask_ptr=None):
        """xq_examples_record_gumbel_device: record_device with the improved-policy weights round(pi' * 2^24) of `gumbel` (a BatchedGumbel
        on a search of the same env) in the visits field"""
        check(self._L.xq_examples_record_gumbel_device(self._h, gumbel._h, mask_ptr))

    def end_games_device(self, ended_ptr, result_ptr):
        """xq_examples_end_games_device: ended u8 [n], result f32 [n] from Red's side"""
        check(self._L.xq_examples_end_games_device(self._h, ended_ptr, result_ptr))

    def discard_device(self, mask_ptr=None):
        check(self._L.xq_examples_discard_device(self._h, mask_ptr))

    def sample_device(self, batch, seed, counter, view, planes_ptr, dtype, policy_ptr, value_ptr=None, q_ptr=None, mask_ptr=None,
                      index_ptr=None):
        check(self._L.xq_examples_sample_device(self._h, int(batch), int(seed), int(counter), view, planes_ptr, dtype, policy_ptr, value_ptr,
                                                q_ptr, mask_ptr, index_ptr))

    def sample_compact_device(self, batch, seed, counter, view, planes_ptr, dtype, actions_ptr, policy_ptr, counts_ptr=None, value_ptr=None,
                              q_ptr=None, index_ptr=None):
        """xq_examples_sample_compact_device: sample_device's rows with compact actions int32 [batch][128] and policy f32 [batch][128]"""
        check(self._L.xq_examples_sample_compact_device(self._h, int(batch), int(seed), int(counter), view, planes_ptr, dtype, actions_ptr,
                                                        policy_ptr, counts_ptr, value_ptr, q_ptr, index_ptr))

    def load_device(self, env, index_ptr):
        """xq_examples_load_device: env e of `env` (a BatchedEnv on the same device) gets the record of ring slot index[e] (int64 [env.n]);
        rows outside the committed examples leave their board"""
        check(self._L.xq_examples_load_device(self._h, env.handle, index_ptr))

    def refresh_device(self, search, index_ptr, status_ptr=None):
        """xq_examples_refresh_device: tree t of `search` (a BatchedSearch on any env of the device) rewrites the targets and q of ring slot
        index[t] (int64 [search.n]); status u8 [search.n] or None"""
        check(self._L.xq_examples_refresh_device(self._h, search._h, index_ptr, status_ptr))

    def refresh_gumbel_device(self, gumbel, index_ptr, status_ptr=None):
        """xq_examples_refresh_gumbel_device: refresh_device with the improved-policy weights of `gumbel` (a begun BatchedGumbel)"""
        check(self._L.xq_examples_refresh_gumbel_device(self._h, gumbel._h, index_ptr, status_ptr))

    def info(self):
        """synchronous: dict of size, capacity, total_committed, pending, dropped, stale"""
        v = [C.c_int64() for _ in range(6)]
        check(self._L.xq_examples_info(self._h, *(C.byref(x) for x in v)))
        return dict(zip(("size", "capacity", "total_committed", "pending", "dropped", "stale"), (x.value for x in v)))

    def get(self, first=0, n=None):
        """synchronous read-back of ring slots [first, first + n): EXAMPLE_DTYPE [n]"""
        n = self.capacity - first if n is None else n
        out = np.zeros(n, EXAMPLE_DTYPE)
        check(self._L.xq_examples_get(self._h, int(first), int(n), ptr(out)))
        return out
