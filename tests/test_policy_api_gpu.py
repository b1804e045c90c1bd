"""GPU tests of the external-policy interface (xq_env_observe_device, xq_env_legal_mask_device, xq_env_policy_step_device) through the
C ABI and TorchEnv: against the oracle (xqo_state, xqo_batch_all_actions, xqo_batch_step), the library's own step and DQN acting, and the
float64 restatement in policy_oracle.py -- on reachable positions, arbitrary boards (the generic path), player bytes 2 and 255 and a grid
whose last CTA is partly empty."""
import numpy as np
import pytest

import policy_oracle as P
from conftest import harvest_positions, random_boards

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def xq():
    import cn_chess_ai_b200 as m
    return m


@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


@pytest.fixture(scope="module")
def mixed(O):
    """reachable positions (both colours to move), arbitrary boards, player bytes 2 / 255; 3,037 boards: the last CTA is partly empty"""
    reach = harvest_positions(O, 500, 4, 7, seed=31)
    arb = random_boards(O, 917, seed=8)
    odd = harvest_positions(O, 120, 1, 11, seed=4)
    odd["player"][:60] = 2
    odd["player"][60:] = 255
    recs = np.concatenate([reach, arb, odd])
    recs["ctr"] = np.arange(len(recs), dtype=np.uint32) * 13 + 5
    assert len(recs) == 3037
    return recs


def _tenv(xq, recs, seed=0, env_id0=0):
    te = xq.TorchEnv(len(recs), seed=seed, env_id0=env_id0)
    te.env.set_boards(recs)
    return te


def _keep(oracle_lib, recs):
    counts, acts = P.oracle_lists(oracle_lib, recs)
    return counts, acts, counts < 128          # the oracle stops its lists at 128 entries


def test_observe_every_dtype_and_view(xq, torch, O, oracle_lib, mixed):
    n = len(mixed)
    st = np.zeros((n, 1260))
    for i in range(n):
        oracle_lib.xqo_state(mixed[i:i + 1].ctypes.data, st[i])
    ab = st.reshape(n, 90, 14).transpose(0, 2, 1)                                   # [n][14][90]
    swap = np.r_[7:14, 0:7]
    side = np.where((mixed["player"] == 1)[:, None, None], ab[:, swap, ::-1], ab)  # channels swapped, s -> 89 - s
    te = _tenv(xq, mixed)
    for dt in (torch.float32, torch.bfloat16, torch.uint8):
        for view, want in (("absolute", ab), ("side", side)):
            planes, aux = te.observe(dtype=dt, view=view)
            got = planes.float().cpu().numpy().reshape(n, 14, 90)
            assert planes.shape == (n, 14, 10, 9) and np.array_equal(got, want), (dt, view)
            a = aux.cpu().numpy()
            assert (a[:, 0] == mixed["player"]).all() and (a[:, 1] == mixed["move_count"]).all()
            assert (a[:, 2] == mixed["red_score"]).all() and (a[:, 3] == mixed["black_score"]).all()
    assert te.env.get_boards().tobytes() == mixed.tobytes()


def test_masks_both_forms_both_views(xq, torch, O, oracle_lib, mixed):
    counts, acts, keep = _keep(oracle_lib, mixed)
    te = _tenv(xq, mixed)
    for view, v in (("absolute", 0), ("side", 1)):
        dense = P.dense_mask(P.policy_indices(mixed, counts, acts, v))
        got = te.legal_mask(packed=False, view=view).cpu().numpy()
        assert got.dtype == bool and not (keep[:, None] & (got != dense)).any(), view
        packed = te.legal_mask(packed=True, view=view).cpu().numpy().view(np.uint32)
        assert not (keep[:, None] & (packed != P.pack_mask(dense))).any(), view
    assert not got[-120:].any()                                                    # player bytes 2 / 255: no action


def test_greedy_equals_dqn_act(xq, O):
    import torch
    recs = harvest_positions(O, 1000, 3, 9, seed=6)
    n = len(recs)
    env = xq.BatchedEnv(n)
    env.set_boards(recs)
    net = xq.DQN(seed=3)
    want, q = xq.act(net, env, eps=0.0, want_q=True)
    te = xq.TorchEnv(env=env)
    scores = torch.from_numpy(np.tile(q[:, :90], 90)).cuda()                      # scores[from * 90 + to] = Q(s)[to]
    r = te.step(scores, pick="greedy", view="absolute", auto_reset=False)
    got = r.actions.cpu().numpy()
    assert np.array_equal((got // 90) << 7 | (got % 90), want.astype(np.int64))
    net.close()


def test_greedy_quantised_scores(xq, torch, O, oracle_lib, mixed):
    counts, acts, keep = _keep(oracle_lib, mixed)
    rng = np.random.default_rng(2)
    for view, v in (("absolute", 0), ("side", 1)):
        for dt in (torch.float32, torch.bfloat16):
            s = (rng.integers(0, 5, (len(mixed), 8100)) / 4).astype(np.float32)    # exact in bf16 too: ties everywhere
            idx = P.policy_indices(mixed, counts, acts, v)
            k = P.greedy(P.listed_scores(s, idx), counts)
            want = np.where(k >= 0, idx[np.arange(len(mixed)), np.maximum(k, 0)], -1)
            te = _tenv(xq, mixed)
            r = te.step(torch.from_numpy(s).cuda().to(dt), pick="greedy", view=view, auto_reset=False)
            got = r.actions.cpu().numpy()
            assert not (keep & (got != want)).any(), (view, dt)


def test_greedy_trajectory_matches_oracle(xq, torch, O, oracle_lib):
    """4,096 envs x 200 plies from the opening, GREEDY on seeded per-ply scores s[from * 90 + to] = a[from] + b[to], auto-reset"""
    n, plies = 4096, 200
    te = xq.TorchEnv(n, seed=5)
    ref = O.new_envs(n)
    g = torch.Generator(device="cuda")
    rows = np.arange(n)
    for p in range(plies):
        g.manual_seed(1000 + p)
        a = torch.rand((n, 90), generator=g, device="cuda")
        b = torch.rand((n, 90), generator=g, device="cuda")
        r = te.step((a[:, :, None] + b[:, None, :]).reshape(n, 8100), pick="greedy", view="absolute", auto_reset=True)
        an, bn = a.cpu().numpy(), b.cpu().numpy()
        counts, acts = P.oracle_lists(oracle_lib, ref)
        frm, to = (acts >> 7).astype(np.int64), (acts & 127).astype(np.int64)
        l = np.where(np.arange(128)[None, :] < counts[:, None], an[rows[:, None], np.minimum(frm, 89)] + bn[rows[:, None], np.minimum(to, 89)], -np.inf)
        k = np.argmax(l, axis=1)
        act = np.where(counts > 0, acts[rows, k], 0xFFFF).astype(np.uint16)
        rew = np.zeros(n, np.int32)
        done, win, cap, valid = (np.zeros(n, np.uint8) for _ in range(4))
        oracle_lib.xqo_batch_step(ref.ctypes.data, n, act, rew, done, win, cap, valid)
        want_idx = np.where(counts > 0, (act >> 7).astype(np.int64) * 90 + (act & 127), -1)
        assert np.array_equal(r.actions.cpu().numpy(), want_idx), p
        for name, w in (("reward", rew), ("done", done), ("winner", win), ("captured", cap), ("valid", valid)):
            assert np.array_equal(getattr(r, name).cpu().numpy(), w), (p, name)
        for i in np.nonzero(done)[0]:                                              # auto-reset keeps the RNG counter
            c = ref[i]["ctr"]
            oracle_lib.xqo_reset(ref[i:i + 1].ctypes.data)
            ref[i]["ctr"] = c
        assert te.env.get_boards().tobytes() == ref.tobytes(), p


def test_sample_against_float64_oracle(xq, torch, O, oracle_lib, mixed):
    counts, acts, keep = _keep(oracle_lib, mixed)
    rng = np.random.default_rng(7)
    seed, id0 = 99, 4000
    u = P.uniform(O.rng_np, seed, np.arange(len(mixed)) + id0, mixed["ctr"])
    for view, v, t in (("absolute", 0, 1.0), ("side", 1, 0.5), ("side", 1, 4.0)):
        s = (rng.standard_normal((len(mixed), 8100)) * 2).astype(np.float32)
        idx = P.policy_indices(mixed, counts, acts, v)
        l = P.listed_scores(s, idx)
        k, _, amb = P.sample(l, counts, t, u)
        want = np.where(k >= 0, idx[np.arange(len(mixed)), np.maximum(k, 0)], -1)
        te = _tenv(xq, mixed, seed=seed, env_id0=id0)
        r = te.step(torch.from_numpy(s).cuda(), pick="sample", temperature=t, view=view, auto_reset=False)
        got, logp = r.actions.cpu().numpy(), r.logp.cpu().numpy()
        assert not (keep & ~amb & (got != want)).any()
        for i in np.nonzero(keep & amb & (got != want))[0]:
            assert got[i] in idx[i, max(k[i] - 1, 0):k[i] + 2]
        kk = np.array([list(idx[i]).index(x) if x >= 0 else -1 for i, x in enumerate(got)])
        fin = keep & (counts > 0)
        assert np.abs(logp[fin] - P.logp_of(l, kk, t)[fin]).max() < 1e-5
        assert (got[counts == 0] == -1).all() and np.isnan(logp[counts == 0]).all()
        vb = r.valid.cpu().numpy()
        assert (vb == (counts > 0)).all()


def test_sample_distribution_rerun_and_sharding(xq, torch, O):
    from scipy import stats
    n = 100_000
    rng = np.random.default_rng(1)
    row = (rng.standard_normal(8100) * 1.5).astype(np.float32)
    scores = torch.from_numpy(row).cuda().expand(n, 8100).contiguous()
    te = xq.TorchEnv(n, seed=42)
    mask = te.legal_mask(view="absolute")[0].cpu().numpy()
    legal = np.nonzero(mask)[0]
    assert len(legal) == 44
    r = te.step(scores, pick="sample", temperature=1.3, view="absolute", auto_reset=False)
    got = r.actions.cpu().numpy()
    p = np.exp((row[legal].astype(np.float64) - row[legal].max()) / 1.3)
    p /= p.sum()
    obs = np.array([(got == i).sum() for i in legal])
    assert obs.sum() == n
    assert stats.chisquare(obs, p * n).pvalue > 1e-4
    # rerun from the same boards: identical actions
    te2 = xq.TorchEnv(n, seed=42)
    assert np.array_equal(te2.step(scores, pick="sample", temperature=1.3, view="absolute").actions.cpu().numpy(), got)
    # two handles splitting the env range via env_id0: the same actions as one handle
    h = 37_501
    ta, tb = xq.TorchEnv(h, seed=42, env_id0=0), xq.TorchEnv(n - h, seed=42, env_id0=h)
    ga = ta.step(scores[:h].contiguous(), pick="sample", temperature=1.3, view="absolute").actions.cpu().numpy()
    gb = tb.step(scores[h:].contiguous(), pick="sample", temperature=1.3, view="absolute").actions.cpu().numpy()
    assert np.array_equal(np.concatenate([ga, gb]), got)


def test_given_equals_step_and_logp(xq, torch, O, oracle_lib, mixed):
    recs = mixed[:-120]                                                          # the library's own step on player bytes 0 / 1 only
    n = len(recs)
    counts, acts, keep = _keep(oracle_lib, recs)
    rng = np.random.default_rng(12)
    s = torch.from_numpy((rng.standard_normal((n, 8100)) * 2).astype(np.float32)).cuda()
    te = _tenv(xq, recs, seed=3)
    sampled = te.step(s, pick="sample", temperature=0.7, view="side", auto_reset=False)
    # GIVEN from the same boards: the sampled actions (same logp), then rejected ones
    given = sampled.actions.clone()
    sel = np.arange(n)
    given_np = given.cpu().numpy()
    idx = P.policy_indices(recs, counts, acts, 1)
    dense = P.dense_mask(idx)
    illegal = np.where(keep, [int(np.nonzero(~dense[i])[0][i % 97]) for i in range(n)], -1)
    given_np = np.where(sel % 5 == 1, -1, np.where(sel % 5 == 2, 8100, np.where(sel % 5 == 3, illegal, given_np)))
    tg = _tenv(xq, recs, seed=3)
    rg = tg.step(s, torch.from_numpy(given_np).cuda(), pick="given", temperature=0.7, view="side", auto_reset=True)
    lp_s, lp_g = sampled.logp.cpu().numpy(), rg.logp.cpu().numpy()
    same = (sel % 5 == 0) | (sel % 5 == 4)
    assert np.array_equal(lp_s[same], lp_g[same], equal_nan=True)
    assert np.isnan(lp_g[~same]).all()
    # the library's step on the converted xq_actions (rejected indices -> XQ_ACTION_NONE)
    flip = P.flip_of(recs, 1)
    legal = same & (given_np >= 0)
    f, t = given_np // 90, given_np % 90
    f, t = np.where(flip, 89 - f, f), np.where(flip, 89 - t, t)
    xa = np.where(legal, (f << 7) | t, 0xFFFF).astype(np.uint16)
    ref = xq.BatchedEnv(n)
    ref.set_boards(recs)
    rew, done, win, cap, valid = ref.step(xa, auto_reset=True)
    for name, w in (("reward", rew), ("done", done), ("winner", win), ("captured", cap), ("valid", valid)):
        assert np.array_equal(getattr(rg, name).cpu().numpy(), w), name
    assert tg.env.get_boards().tobytes() == ref.get_boards().tobytes()
    assert (rg.valid.cpu().numpy()[~same] == 0).all()
    # without scores: checked and applied, no logp
    tg2 = _tenv(xq, recs, seed=3)
    r2 = tg2.step(None, torch.from_numpy(given_np).cuda(), pick="given", view="side", auto_reset=True)
    assert tg2.env.get_boards().tobytes() == ref.get_boards().tobytes() and np.isnan(r2.logp.cpu().numpy()).all()


def test_player_bytes_and_nonfinite(xq, torch, O, oracle_lib, mixed):
    odd = mixed[-120:]
    te = _tenv(xq, odd)
    s = torch.randn((120, 8100), device="cuda")
    r = te.step(s, pick="sample", view="side", auto_reset=False)
    assert (r.actions.cpu().numpy() == -1).all() and (r.valid.cpu().numpy() == 0).all() and np.isnan(r.logp.cpu().numpy()).all()
    assert (r.captured.cpu().numpy() == 0).all() and te.env.get_boards().tobytes() == odd.tobytes()
    # non-finite scores on reachable boards
    recs = mixed[:2000]
    counts, acts, _ = _keep(oracle_lib, recs)
    idx = P.policy_indices(recs, counts, acts, 1)
    first = idx[:, 0]
    for pick in ("greedy", "sample"):
        s = torch.full((2000, 8100), float("-inf"), device="cuda")
        s[:, ::2] = float("nan")
        r = _tenv(xq, recs).step(s, pick=pick, view="side", auto_reset=False)
        assert np.array_equal(r.actions.cpu().numpy(), first) and np.isnan(r.logp.cpu().numpy()).all()
    # +inf is clamped to FLT_MAX: the first +inf in list order wins GREEDY and SAMPLE (probability ~1); one NaN among finite scores never plays
    last = idx[np.arange(2000), counts.astype(np.int64) - 1]
    s = torch.zeros((2000, 8100), device="cuda")
    rows = torch.arange(2000, device="cuda")
    s[rows, torch.from_numpy(first).cuda()] = float("nan")
    s[rows, torch.from_numpy(last).cuda()] = float("inf")
    for pick in ("greedy", "sample"):
        r = _tenv(xq, recs).step(s, pick=pick, view="side", auto_reset=False)
        assert np.array_equal(r.actions.cpu().numpy(), last)
        assert np.abs(r.logp.cpu().numpy()).max() < 1e-6
    # the temperature must be finite and > 0 for SAMPLE and whenever logp is computed
    te = xq.TorchEnv(64)
    s = torch.zeros((64, 8100), device="cuda")
    for t in (0.0, -1.0, float("nan"), float("inf")):
        with pytest.raises(xq.XQError):
            te.step(s, pick="sample", temperature=t)
        with pytest.raises(xq.XQError):
            te.step(s, pick="greedy", temperature=t)                            # TorchEnv always asks for logp
    a = torch.zeros(64, dtype=torch.int64, device="cuda")
    te.step(None, a, pick="given", temperature=0.0)                              # no scores: no logp, no temperature
    with pytest.raises(ValueError):
        te.step(s[:, :100], pick="greedy")
    with pytest.raises(ValueError):
        te.step(s.to(torch.float16), pick="greedy")
