"""The FP64 restatement of the acting path's Q (tests/act_oracle.py) against the oracle's state and network (xqo_state, xqo_nn_forward),
and its error bound at the reference initialisation.  No GPU."""
import numpy as np

import act_oracle as AO
from conftest import harvest_positions, random_boards, recs_from_codes

LA = np.array([1260, 128, 8100], np.int32)


def ref_params(seed):
    rng = np.random.default_rng(seed)
    return rng.uniform(-0.05, 0.05, 1260 * 128 + 128 * 8100), rng.uniform(-0.05, 0.05, 128 + 8100)


def full_boards(O, m, seed):
    """all 90 squares occupied by random pieces: the largest layer-0 sums"""
    rng = np.random.default_rng(seed)
    return recs_from_codes(O, rng.integers(1, 15, (m, 90)).astype(np.uint8), np.zeros((m, 4), np.int32))


def test_fp64_q_matches_the_oracle_network(O, oracle_lib):
    recs = np.concatenate([harvest_positions(O, 64, 3, 25, seed=5), random_boards(O, 64, 8), full_boards(O, 16, 9), O.new_envs(2)])
    codes = AO.codes(recs)
    for i in (0, 70, 150, len(recs) - 1):
        assert (codes[i] == O.codes_of(recs[i])).all()
    for w, b in (ref_params(1), (ref_params(2)[0] * 30, ref_params(2)[1] * 30)):
        q, h = AO.forward(recs, w, b)
        st, qq = np.zeros(1260), np.zeros(8100)
        x, occ = AO.onehot(recs)
        for i in range(len(recs)):
            oracle_lib.xqo_state(recs[i:i + 1].ctypes.data, st)
            assert (x[i].toarray()[0] == st).all() and occ[i] == int(st.sum()), i
            oracle_lib.xqo_nn_forward(LA, 3, w, b, st, qq)
            assert np.abs(q[i] - qq[:96]).max() <= 1e-12, i


def test_code_15_selects_nothing(O):
    """the device sanitises code 15 (no channel in getStateRepresentation); the restatement does the same"""
    c = np.zeros((1, 90), np.uint8); c[0, [0, 44, 89]] = [15, 3, 15]
    x, occ = AO.onehot(recs_from_codes(O, c, np.zeros((1, 4), np.int32)))
    assert occ[0] == 1 and x.nnz == 1 and x.indices[0] == 44 * 14 + 2


def test_quant_shift_matches_the_device_function(hostsim):
    """k of the bound is the k of xq_act_quant.cuh (compiled for the host) for the weight versions the GPU tests use"""
    w, b = ref_params(3)
    versions = [(w, b), (w * 1e-3, b * 1e-3), (w * 30, b * 30)]
    wb = b.copy(); wb[127] = 40.0; versions.append((w, wb))
    wl = w.copy(); wl[127 * 1260 + 1259] = -40.0; versions.append((wl, b))
    for wv, bv in versions:
        W0, b0, _, _ = AO.layers(wv, bv)
        flat = np.concatenate([W0.T.ravel(), b0]).astype(np.float32)
        q = np.zeros(flat.size, np.int32)
        assert AO.act_quant_shift(wv, bv) == hostsim.hs_act_quant(flat.ctypes.data, flat.size, q.ctypes.data)
    assert AO.act_quant_shift(w, b) == 27


def test_bf16_split_of_w1():
    rng = np.random.default_rng(0)
    v = rng.uniform(-0.05, 0.05, 100000)
    lo, dW = AO.w1_split(v)
    hi = v - lo - dW
    assert (AO.bf16(hi) == hi.astype(np.float32)).all() and (AO.bf16(lo) == lo.astype(np.float32)).all()
    assert np.abs(v - hi).max() <= 2.0 ** -8 * np.abs(v).max() and (np.abs(dW) <= 2.0 ** -17 * np.abs(v) + 2.0 ** -24 * np.abs(v)).all()
    assert AO.bf16(np.float32(1.0 + 2.0 ** -8)) == 1.0 and AO.bf16(np.float32(1.0 + 3 * 2.0 ** -8)) == np.float32(1.0 + 2.0 ** -6)  # ties to even


def test_bound_at_the_reference_initialisation(O):
    """the bound is no looser than the 2e-5 the suite used before, on reachable, arbitrary and full boards"""
    w, b = ref_params(4)
    recs = np.concatenate([harvest_positions(O, 256, 4, 30, seed=6), random_boards(O, 256, 10), O.new_envs(1)])
    bnd = AO.bound(recs, w, b)
    assert bnd.max() < 2e-5 and bnd.min() > 2e-6, (bnd.min(), bnd.max())
    full = AO.bound(full_boards(O, 64, 11), w, b)
    assert full.max() < 4e-5
    big = AO.bound(recs, w * 30, b * 30)
    assert (big > bnd).all()


def test_greedy_check_flags_a_wrong_choice(O, oracle_lib):
    """the action check of the GPU tests: the FP64 first maximum passes, another action fails unless it is near-tied"""
    from policy_oracle import oracle_lists
    w, b = ref_params(5)
    recs = harvest_positions(O, 128, 2, 20, seed=7)
    q, _ = AO.forward(recs, w, b)
    bnd = AO.bound(recs, w, b)
    counts, acts = oracle_lists(oracle_lib, recs)
    pos = np.arange(128)[None, :] < counts[:, None]
    tq = np.where(pos, np.take_along_axis(q, np.minimum(acts.astype(np.int64) & 127, 95), axis=1), -np.inf)
    best = acts[np.arange(len(recs)), np.argmax(tq, axis=1)]
    bad, near, checked = AO.greedy_check(counts, acts, best, q, bnd)
    assert len(bad) == 0 and checked == len(recs) and near < checked // 10
    worst = acts[np.arange(len(recs)), np.argmin(np.where(pos, tq, np.inf), axis=1)]
    bad, _, _ = AO.greedy_check(counts, acts, worst, q, bnd)
    assert len(bad) == len(recs)
