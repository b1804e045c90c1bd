"""The acting path (xq_dqn_act, xq_selfplay_collect) against the FP64 network entry by entry, at the benchmarked 65,536 envs and at the
edges of its kernels: the persistent tile loop of q90_gemm_kernel, the carried fixed-point layer-0 sums, the per-version scale of the
fixed-point table, several env handles on one network and the replay ring.  Every entry of Q(s)[0..95] must lie within the error bound
of tests/act_oracle.py; with eps = 0 the chosen action must be the FP64 first maximum of Q[to] over the oracle's list, or one of the
actions near-tied with it within the bound.  Each case prints its worst |dQ|, its worst |dQ| / bound and its near ties."""
import numpy as np
import pytest

import act_oracle as AO
from conftest import random_boards, recs_from_codes
from policy_oracle import oracle_lists

pytestmark = pytest.mark.gpu
LAYERS = [1260, 128, 8100]
N_W0 = 1260 * 128


@pytest.fixture(scope="module")
def xq():
    import cn_chess_ai_b200 as m
    return m


def rand_params(seed):
    rng = np.random.default_rng(seed)
    return rng.uniform(-0.05, 0.05, 1260 * 128 + 128 * 8100), rng.uniform(-0.05, 0.05, 128 + 8100)


def pack(codes):
    c = np.zeros((len(codes), 96), np.uint32)
    c[:, :90] = codes
    return (c.reshape(-1, 12, 8) << (4 * np.arange(8, dtype=np.uint32))).sum(axis=2, dtype=np.uint32)


def check_q(q, recs, w, b, tag):
    """every entry of the device Q(s)[0..95] within the bound of the FP64 Q; returns (FP64 Q, bound)"""
    q64, h = AO.forward(recs, w, b)
    bnd = AO.bound(recs, w, b, h)
    err = np.abs(q[:, :96].astype(np.float64) - q64)
    bad = np.argwhere(err > bnd)
    assert len(bad) == 0, (tag, len(bad), [(int(i), int(o), float(err[i, o]), float(bnd[i, o])) for i, o in bad[:5]])
    print(f"[act-fp64] {tag}: n={len(recs)} worst |dQ|={err.max():.3e} worst |dQ|/bound={(err / bnd).max():.3f} max bound={bnd.max():.3e}")
    return q64, bnd


def check_greedy(L, recs, actions, q64, bnd, tag):
    counts, acts = oracle_lists(L, recs)
    bad, near, checked = AO.greedy_check(counts, acts, actions, q64, bnd)
    assert len(bad) == 0, (tag, bad[:10])
    print(f"[act-fp64] {tag}: greedy actions checked={checked} near ties={near}")
    assert near <= 0.01 * checked, (tag, near, checked)
    return near


def mixed_env(xq, O, n, seed):
    """mid-game positions from device rollouts, ~2 % arbitrary boards (generic act kernel) and a few finished boards"""
    env = xq.BatchedEnv(n, seed=seed)
    env.rollout_random(30 + seed % 40)
    recs = env.get_boards()
    rng = np.random.default_rng(seed)
    perm = rng.permutation(n)
    m = n // 50
    if m:
        recs[perm[:m]] = random_boards(O, m, seed)
    fin = perm[m:m + n // 2000 + (n >= 100)]
    recs["move_count"][fin[::2]] = 200                       # the move cap
    c = AO.codes(recs[fin[1::2]])
    c[c == 8] = 0                                            # the Black General taken
    recs["sq"][fin[1::2]] = pack(c)
    env.set_boards(recs)
    return env, recs


@pytest.mark.parametrize("n", [1, 127, 129, 18944, 18945, 37889, 65536, 65613])
def test_q_and_greedy_choice_across_the_persistent_tile_loop(xq, O, oracle_lib, n):
    """18,944 envs = 148 tiles (one per CTA); 18,945: CTA 0 takes a second 1-row tile; 37,889: three tiles on CTA 0, so the A-ring and
    accumulator stages are reused with flipped phases; 65,536: the benchmarked size; 65,613: a partial last tile"""
    w, b = rand_params(40)
    net = xq.DQN(LAYERS); net.set_params(w, b)
    env, recs = mixed_env(xq, O, n, seed=n % 997)
    actions, q = xq.act(net, env, 0.0, want_q=True)
    assert env.get_boards().tobytes() == recs.tobytes()
    q64, bnd = check_q(q, recs, w, b, f"tiles n={n}")
    check_greedy(oracle_lib, recs, actions, q64, bnd, f"tiles n={n}")


def test_carried_sums_at_scale(xq, O):
    """65,613 envs, 30 plies of act + step (eps 0.3, auto-reset): the sums are carried from ply to ply (l0_act_kernel).  At ply 10 a
    set_boards leaves some envs exactly 4 squares away from the board their sum belongs to (still carried) and others exactly 5 (gathered
    again); the changed squares include 0, 88 and 89 (word 11 holds only 88 and 89)."""
    n, plies, eps = 65613, 30, 0.3
    w, b = rand_params(41)
    net = xq.DQN(LAYERS); net.set_params(w, b)
    env = xq.BatchedEnv(n, seed=5, env_id0=7)
    rng = np.random.default_rng(5)
    prev = None
    for p in range(plies):
        if p == 10:
            recs = env.get_boards()
            for k, sel in ((4, np.arange(3, n, 13)), (5, np.arange(7, n, 13))):
                new = prev[sel].copy()
                c = AO.codes(new)
                extra = np.stack([rng.choice(np.arange(1, 88), k - 3, replace=False) for _ in sel])
                sq = np.concatenate([np.tile([0, 88, 89], (len(sel), 1)), extra], axis=1)
                r = np.arange(len(sel))[:, None]
                c[r, sq] = c[r, sq] % 14 + 1                      # a different piece (or a piece on an empty square)
                new["sq"] = pack(c)
                assert ((AO.codes(new) != AO.codes(prev[sel])).sum(axis=1) == k).all()
                recs[sel] = new
            env.set_boards(recs)
        actions, q = xq.act(net, env, eps, want_q=True)
        if p % 5 == 0 or p == plies - 1:
            check_q(q, env.get_boards(), w, b, f"carried ply {p}")
        prev = env.get_boards()
        env.step(actions, auto_reset=True)


def boards_selecting_the_last_row(O, recs, m):
    """m boards with a Black piece of code 14 on square 89: they select input 1259, the last row of W0^T"""
    out = recs[:m].copy()
    c = AO.codes(out)
    c[:, 89] = 14
    out["sq"] = pack(c)
    return out


def test_weight_versions_on_one_handle(xq, O, oracle_lib):
    """The fixed-point scale k follows max |W0|, |b0| per weight version (act_quant_max_kernel's grid-stride reduction over W0^T then b0,
    the alternating max slots).  Each version on one handle: within the bound of FP64 and bit for bit the Q of a fresh handle."""
    n = 4096
    env, recs = mixed_env(xq, O, n, seed=77)
    recs[:256] = boards_selecting_the_last_row(O, recs, 256)
    env.set_boards(recs)
    w, b = rand_params(42)
    versions = [("reference init", w, b)]
    w1, b1 = w.copy(), b.copy(); w1[:N_W0] *= 1e-3; b1[:128] *= 1e-3
    versions.append(("W0, b0 x 1e-3", w1, b1))
    b2 = b.copy(); b2[127] = 40.0
    versions.append(("b0[127] = +40", w, b2))
    w3 = w.copy(); w3[127 * 1260 + 1259] = -40.0
    versions.append(("W0[127, 1259] = -40", w3, b))
    w4, b4 = w.copy(), b.copy(); w4[:N_W0] *= 30; b4[:128] *= 30
    versions.append(("W0, b0 x 30", w4, b4))
    versions.append(("reference init again", w, b))
    net = xq.DQN(LAYERS)
    for tag, wv, bv in versions:
        net.set_params(wv, bv)
        a, q = xq.act(net, env, 0.0, want_q=True)
        fresh = xq.DQN(LAYERS); fresh.set_params(wv, bv)
        af, qf = xq.act(fresh, env, 0.0, want_q=True)
        assert np.array_equal(q.view(np.uint32), qf.view(np.uint32)) and (a == af).all(), tag
        q64, bnd = check_q(q, recs, wv, bv, f"version {tag}")
        if tag.startswith("reference"):
            assert bnd.max() < 2e-5
            check_greedy(oracle_lib, recs, a, q64, bnd, f"version {tag}")
    # the worst case the scale is chosen for: all 90 squares occupied, every selected row +M at hidden unit 5 and b0[5] = +M, with
    # 92 M just below 2^4 (k = 26): the sum reaches 91/92 of 2^30 and h = tanh(91 M) must saturate at +1 as in FP64, not wrap to -1
    M = np.float32(16.0 / 92.0)
    while np.float32(92.0) * M >= np.float32(16.0):
        M = np.nextafter(M, np.float32(0))
    wf, bf = w.copy(), b.copy()
    wf[5 * 1260:6 * 1260] = float(M); bf[5] = float(M)
    assert AO.act_quant_shift(wf, bf) == 26
    rng = np.random.default_rng(9)
    full = recs_from_codes(O, rng.integers(1, 15, (256, 90)).astype(np.uint8), np.zeros((256, 4), np.int32))
    envf = xq.BatchedEnv(256, seed=3)
    envf.set_boards(full)
    net.set_params(wf, bf)
    a, q = xq.act(net, envf, 0.0, want_q=True)
    fresh = xq.DQN(LAYERS); fresh.set_params(wf, bf)
    _, qf = xq.act(fresh, envf, 0.0, want_q=True)
    assert np.array_equal(q.view(np.uint32), qf.view(np.uint32))
    _, h = AO.forward(full, wf, bf)
    assert (h[:, 5] > 1 - 1e-12).all()
    check_q(q, full, wf, bf, "full boards at the bound of the scale")


def stepwise(xq, O, L, net, twin, ref, plies, eps, ring_rows):
    """the step-by-step path on a twin env (GPU act on the same Q and draws + oracle rules) against the transitions of a collect"""
    n = len(ref)
    for p in range(plies):
        actions = xq.act(net, twin, eps)
        before = ref.copy()
        r0 = np.zeros(n, np.int32); d0, w0, c0, v0 = (np.zeros(n, np.uint8) for _ in range(4))
        L.xqo_batch_step(ref.ctypes.data, n, actions, r0, d0, w0, c0, v0)
        t = ring_rows[p]
        assert (t["action"] == actions).all() and (t["reward"] == r0).all(), p
        assert t["s"].tobytes() == before["sq"].tobytes() and t["s2"].tobytes() == ref["sq"].tobytes(), p
        for i in np.nonzero(d0)[0]:
            L.xqo_reset(ref[i:i + 1].ctypes.data)
        twin.step(actions, auto_reset=True)
    assert twin.get_boards().tobytes() == ref.tobytes()


def test_one_network_several_env_handles(xq, O, oracle_lib):
    """A (20,000) collect -> B (30,000) act -> A collect -> C (129) act -> B collect on one network: the acting buffers grow under A's
    two-stream halves (their tensor maps must follow the new buffers).  After each call the actions / transitions equal the step-by-step
    path on a twin env acting through a second network with the same parameters, and Q is within the bound of FP64 and bit for bit the
    twin's."""
    w, b = rand_params(43)
    net = xq.DQN(LAYERS); net.set_params(w, b)
    twin_net = xq.DQN(LAYERS); twin_net.set_params(w, b)
    plies, eps = 4, 0.3
    sizes = {"A": 20000, "B": 30000, "C": 129}
    envs = {k: xq.BatchedEnv(m, seed=11 + m % 7, env_id0=m) for k, m in sizes.items()}
    twins = {k: xq.BatchedEnv(m, seed=11 + m % 7, env_id0=m) for k, m in sizes.items()}
    refs = {k: O.new_envs(m) for k, m in sizes.items()}
    for step, (k, call) in enumerate([("A", "collect"), ("B", "act"), ("A", "collect"), ("C", "act"), ("B", "collect")]):
        env, twin, ref, m = envs[k], twins[k], refs[k], sizes[k]
        if call == "collect":
            rb = xq.ReplayBuffer(m * plies)
            xq.collect(net, env, rb, plies, eps, train_done=True)
            env.sync()
            stepwise(xq, O, oracle_lib, twin_net, twin, ref, plies, eps, rb.get(0, m * plies).reshape(plies, m))
            assert env.get_boards().tobytes() == ref.tobytes(), step
        a, q = xq.act(net, env, eps, want_q=True)
        at, qt = xq.act(twin_net, twin, eps, want_q=True)
        assert (a == at).all() and np.array_equal(q.view(np.uint32), qt.view(np.uint32)), step
        check_q(q, env.get_boards(), w, b, f"handles step {step} {k} {call}")


def test_collect_refuses_a_ring_smaller_than_one_ply(xq):
    """every env of a ply writes its own ring slot at once: a ring of fewer slots than envs is refused before anything runs"""
    n = 1000
    w, b = rand_params(44)
    net = xq.DQN(LAYERS); net.set_params(w, b)
    env = xq.BatchedEnv(n, seed=2)
    rb = xq.ReplayBuffer(n - 1)
    seed_batch = np.zeros(300, xq.TRANSITION_DTYPE)
    seed_batch["reward"] = np.arange(300); seed_batch["action"] = 7
    rb.insert(seed_batch)
    env.step(xq.act(net, env, 0.5), auto_reset=True)
    ring, info, boards, stats = rb.get(), rb.info(), env.get_boards(), env.stats()
    with pytest.raises(xq.XQError):
        xq.collect(net, env, rb, 3, 0.1)
    env.sync()
    assert rb.get().tobytes() == ring.tobytes() and rb.info() == info
    assert env.get_boards().tobytes() == boards.tobytes() and env.stats().tobytes() == stats.tobytes()
    ok = xq.ReplayBuffer(n)                                  # one ply exactly fits
    xq.collect(net, env, ok, 2, 0.1)
    assert ok.info() == (n, n, 2 * n)
