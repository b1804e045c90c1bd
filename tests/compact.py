"""numpy restatement of the compact action lists (include/xq.h: XQ_COMPACT_ACTIONS), shared by test_compact_cpu.py and
test_compact_gpu.py: the oracle's reference-ordered list (xqo_batch_all_actions, the first 128 actions) mapped to the frame of the view."""
import numpy as np

import policy_oracle as P


def compact_lists(L, recs, view):
    """(actions int32 [n, 128]: policy indices of list entries k in the frame of `view`, -1 past the count; counts uint8 [n])"""
    counts, acts = P.oracle_lists(L, recs)
    return P.policy_indices(recs, counts, acts, view).astype(np.int32), counts


def gather(dense, actions):
    """compact rows C[k] = D[actions[k]] of dense rows D (entries past the count are left as D[0]: never read)"""
    return np.take_along_axis(dense, np.maximum(actions, 0).astype(np.int64), axis=1)


def garbage_dense(rng, n, nan_frac=0.05, inf_frac=0.02):
    """dense f32 score rows: normal noise with NaN, +inf and -inf sprinkled in (only the listed entries are read)"""
    d = rng.normal(0.0, 2.0, (n, 8100)).astype(np.float32)
    u = rng.random((n, 8100))
    d[u < nan_frac] = np.nan
    d[(u >= nan_frac) & (u < nan_frac + inf_frac)] = np.inf
    d[(u >= nan_frac + inf_frac) & (u < nan_frac + 2 * inf_frac)] = -np.inf
    return d
