"""numpy restatement of the external-policy interface (include/xq.h: xq_env_observe_device, xq_env_legal_mask_device,
xq_env_policy_step_device), shared by test_policy_api_cpu.py and test_policy_api_gpu.py.  Lists come from the oracle
(xqo_batch_all_actions); everything else is spelled out here in float64."""
import numpy as np

FLT_MAX = float(np.finfo(np.float32).max)


def oracle_lists(L, recs):
    n = len(recs)
    counts = np.zeros(n, np.uint8)
    acts = np.zeros((n, 128), np.uint16)
    L.xqo_batch_all_actions(recs.ctypes.data, n, counts, acts)
    acts[np.arange(128)[None, :] >= counts[:, None]] = 0xFFFF
    return counts, acts


def flip_of(recs, view):
    return (view == 1) & (recs["player"] == 1)


def policy_indices(recs, counts, acts, view):
    """[n, 128] int64 policy indices of the reference-ordered lists in the frame of `view`, -1 past the count"""
    frm, to = (acts >> 7).astype(np.int64), (acts & 127).astype(np.int64)
    idx = np.where(flip_of(recs, view)[:, None], (89 - frm) * 90 + (89 - to), frm * 90 + to)
    idx[np.arange(128)[None, :] >= counts[:, None]] = -1
    return idx


def dense_mask(idx):
    n = len(idx)
    m = np.zeros((n, 8100 + 1), bool)
    m[np.repeat(np.arange(n), idx.shape[1]), idx.ravel()] = True      # -1 lands in the spare column
    return m[:, :8100]


def pack_mask(dense):
    bits = np.zeros((len(dense), 254 * 32), np.uint8)
    bits[:, :8100] = dense
    return np.packbits(bits, axis=1, bitorder="little").view("<u4")


def clean(x):
    x = np.asarray(x, np.float64)
    return np.where(np.isnan(x), -np.inf, np.minimum(x, FLT_MAX))


def listed_scores(scores, idx):
    """cleaned scores of the listed actions [n, 128], -inf past the count"""
    l = clean(np.take_along_axis(scores, np.maximum(idx, 0), axis=1))
    return np.where(idx >= 0, l, -np.inf)


def greedy(l, counts):
    """first maximum in list order (argmax returns the first); -1 for an empty list"""
    return np.where(counts > 0, np.argmax(l, axis=1), -1)


def uniform(rng_np, seed, env_ids, ctrs):
    x = rng_np(seed, env_ids, ctrs)
    return (x >> np.uint64(40)).astype(np.float32).astype(np.float64) * 2.0 ** -24


def sample(l, counts, t, u):
    """SAMPLE in float64: (k, logp of k, ambiguous) -- ambiguous where u*S lies within 1e-5*S of a boundary of the cumulative sum
    (there either neighbour is a correct float32 answer)"""
    n = len(l)
    m = l.max(axis=1)
    fin = np.isfinite(m)
    with np.errstate(invalid="ignore", over="ignore"):
        e = np.where(np.isfinite(l) & fin[:, None], np.exp((l - np.where(fin, m, 0)[:, None]) / t), 0.0)
    cum = np.cumsum(e, axis=1)
    s = cum[:, -1]
    thr = u * s
    k = np.argmax(cum > thr[:, None], axis=1)
    prev = np.where(k > 0, cum[np.arange(n), np.maximum(k - 1, 0)], 0.0)
    amb = (np.abs(cum[np.arange(n), k] - thr) < 1e-5 * s) | (np.abs(prev - thr) < 1e-5 * s)
    k = np.where(fin, k, 0)
    k = np.where(counts > 0, k, -1)
    return k, logp_of(l, k, t), amb


def logp_of(l, k, t):
    n = len(l)
    m = l.max(axis=1)
    fin = np.isfinite(m)
    with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
        e = np.where(np.isfinite(l) & fin[:, None], np.exp((l - np.where(fin, m, 0)[:, None]) / t), 0.0)
        lk = l[np.arange(n), np.maximum(k, 0)]
        lp = (lk - m) / t - np.log(e.sum(axis=1))
    return np.where(fin & (k >= 0), lp, np.nan)
