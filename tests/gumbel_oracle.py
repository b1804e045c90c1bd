"""numpy restatement of the Gumbel root search (include/xq.h: xq_gumbel_*), shared by test_gumbel_cpu.py and test_gumbel_gpu.py: the
Gumbel draw, the considered set, the Sequential Halving sequence, the completed Q, sigma and the improved policy, the root rule with
in-flight counts and its fallback, and the action to play.  The rounded arithmetic is spelled out in np.float32 in the stated operation
order, so that it matches the device bit for bit; logf / expf are numpy's.  GumbelTree extends search_leaves_oracle.LeavesTree with the
Gumbel root rule of xq_gumbel_select_device."""
import math

import numpy as np

import search_leaves_oracle as SL

F32 = np.float32
FLT_MIN = np.finfo(np.float32).tiny
GUMBEL_WORD = 128


def rng_np(seed, env, ctr):
    """xq_rng on uint64 arrays (wrapping arithmetic)"""
    with np.errstate(over="ignore"):
        z = (np.uint64(seed) + np.asarray(env, np.uint64) * np.uint64(0x9E3779B97F4A7C15)
             + np.asarray(ctr, np.uint64) * np.uint64(0xD1B54A32D192ED03))
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))


def gumbel_u(base, n):
    """u_k = (f + 0.5) * 2^-24, f = bits 40..63 of xq_rng(base, k, 128), k = 0 .. n - 1 (exact in f32)"""
    f = (rng_np(base, np.arange(n, dtype=np.uint64), GUMBEL_WORD) >> np.uint64(40)).astype(np.float64)
    return ((f + 0.5) * 2.0 ** -24).astype(F32)


def gumbel_draw(base, n):
    """g_k = -log(-log u_k) in f32 (numpy's log)"""
    u = gumbel_u(base, n)
    return (-np.log(-np.log(u))).astype(F32)


def considered(key, m):
    """bool [n]: the top min(m, n) keys, ties to the smaller index (a stable sort of -key)"""
    key = np.asarray(key, F32)
    order = np.argsort(-key.astype(np.float64), kind="stable")
    out = np.zeros(len(key), bool)
    out[order[:min(m, len(key))]] = True
    return out


def sequence(m, n):
    """mctx's get_sequence_of_considered_visits(m, n), restated from its description"""
    if m <= 1:
        return list(range(n))
    log2max = int(math.ceil(math.log2(m)))
    seq, visits, mc = [], [0] * m, m
    while len(seq) < n:
        extra = max(1, int(n / (log2max * mc)))
        for _ in range(extra):
            seq.extend(visits[:mc])
            for i in range(mc):
                visits[i] += 1
        mc = max(2, mc // 2)
    return seq[:n]


def completed_q(N, W, P, vhat):
    """(q completed [n], v_mix): q_k = W_k / N_k when visited, else v_mix; sums in list order in f32"""
    N = np.asarray(N, np.int64)
    W, P = np.asarray(W, F32), np.asarray(P, F32)
    sn, sp, sq = 0, F32(0), F32(0)
    for k in range(len(N)):
        if N[k] > 0:
            sn += int(N[k])
            p = F32(max(P[k], FLT_MIN))
            sp = F32(sp + p)
            sq = F32(sq + F32(p * F32(W[k] / F32(N[k]))))
    vm = F32(F32(F32(vhat) + F32(F32(sn) * F32(sq / sp))) / F32(sn + 1)) if sn > 0 else F32(vhat)
    with np.errstate(divide="ignore", invalid="ignore"):
        q = np.where(N > 0, W / N.astype(F32), vm).astype(F32)
    return q, vm


def sigma(N, W, P, vhat, c_visit, c_scale):
    """sigma [n] = ((c_visit + max N) * c_scale) * (q - min) / max(max - min, 1e-8) of the completed q"""
    q, _ = completed_q(N, W, P, vhat)
    mn, mx = q.min(), q.max()
    qh = ((q - mn).astype(F32) / max(F32(mx - mn), F32(1e-8))).astype(F32)
    return (F32(F32(F32(c_visit) + F32(int(np.max(N)))) * F32(c_scale)) * qh).astype(F32)


def root_scores(N, W, P, g, logit, vhat, c_visit, c_scale):
    """(z = logit + sigma, score = (g + logit) + sigma)"""
    sg = sigma(N, W, P, vhat, c_visit, c_scale)
    logit, g = np.asarray(logit, F32), np.asarray(g, F32)
    return (logit + sg).astype(F32), ((g + logit).astype(F32) + sg).astype(F32)


def improved_policy(z):
    """(pi' [n], integer weights round-half-even(pi' * 2^24)): exp(z - max) / S, S summed in list order"""
    z = np.asarray(z, F32)
    e = np.exp((z - z.max()).astype(F32)).astype(F32)
    s = F32(0)
    for x in e:
        s = F32(s + x)
    p = (e / s).astype(F32)
    return p, np.rint((p * F32(2.0 ** 24)).astype(F32)).astype(np.int64)


def argmax_first(score, mask):
    """the largest score among mask, first index on ties; -1 if mask is empty"""
    idx = np.nonzero(mask)[0]
    if len(idx) == 0:
        return -1
    s = np.asarray(score, F32)[idx]
    return int(idx[int(np.argmax(s))])


def pick(cons, cnt, score, target):
    """the root rule: considered edges with cnt == target, else those with the fewest cnt; the largest score, first index on ties"""
    cons, cnt = np.asarray(cons, bool), np.asarray(cnt, np.int64)
    want = target if (cons & (cnt == target)).any() else cnt[cons].min()
    return argmax_first(score, cons & (cnt == want))


def action(cons, nv, score):
    """the considered edge with the most visits this move, then the largest score, then the first index; -1 when none has a visit"""
    cons, nv = np.asarray(cons, bool), np.asarray(nv, np.int64)
    live = cons & (nv > 0)
    if not live.any():
        return -1
    return argmax_first(score, live & (nv == nv[live].max()))


class GumbelTree(SL.LeavesTree):
    """a LeavesTree whose root rule during a Gumbel search is set by begin(state, ...) with the device's g and logit (state of
    xq_gumbel_get: gumbel, logit, considered, n0, root_value, m)"""

    def begin(self, st, n_sims, c_visit, c_scale):
        self.gs = st
        self.n_sims, self.c_visit, self.c_scale, self.done = n_sims, c_visit, c_scale, 0

    def root_stats(self):
        ne = len(self.act[0])
        g, lg = self.gs["gumbel"][:ne], self.gs["logit"][:ne]
        z, sc = root_scores(self.N[0], self.W[0], self.P[0], g, lg, self.gs["root_value"], self.c_visit, self.c_scale)
        return z, sc, self.gs["considered"][:ne], (self.N[0] - self.gs["n0"][:ne]).astype(np.int64)

    def select_gumbel(self, L, c_puct, fpu, vl):
        """select_leaves with the Gumbel root rule at the root"""
        inflight, ended, out = {}, set(), []
        z, sc, cons, nv = self.root_stats() if self.expanded[0] and not self.status[0] else (None,) * 4
        seq = sequence(self.gs["m"], self.n_sims)
        for d in range(L):
            j, path = 0, []
            while self.expanded[j] and not self.status[j]:
                ne = len(self.act[j])
                c = np.array([inflight.get((j, e), 0) for e in range(ne)], np.int64)
                if j == 0:
                    k = pick(cons, nv + c, sc, seq[self.done + d])
                else:
                    k = int(np.argmax(SL.puct_vl(self.P[j], self.N[j], self.W[j], c, vl, c_puct, fpu, self.visits[j], int(c.sum()))))
                path.append((j, k))
                if self.child[j][k] >= 0:
                    j = int(self.child[j][k])
                    continue
                j = self._make_child(j, k)
                break
            for key in path:
                inflight[key] = inflight.get(key, 0) + 1
            dup = not self.expanded[j] and self.status[j] == 0 and j in ended
            ended.add(j)
            out.append((j, SL.DUPLICATE if dup else self.status[j]))
        self.done += L
        return out

    def gumbel_root(self, view):
        """(pi' [8100] in the frame of view, action or -1, pi' in list order)"""
        pol = np.zeros(8100, F32)
        if self.gs["m"] == 0:
            return pol, -1, None
        z, sc, cons, nv = self.root_stats()
        p, _ = improved_policy(z)
        flip = view == 1 and self.rec[0]["player"] == 1
        idx = np.where(flip, 8099 - self.act[0], self.act[0])
        pol[idx] = p
        k = action(cons, nv, sc)
        return pol, (int(idx[k]) if k >= 0 else -1), p



def improved_policy64(N, W, P, logit, vhat, c_visit, c_scale):
    """(pi' in float64, a per-entry bound on |pi'_f32 - pi'_64|) of one root from its edges' N, W, P, the stored logits and the root
    value.  The float64 restatement is completed_q / sigma / improved_policy without rounding; the bound follows their f32 operation
    order with u = 2^-24 per rounding:
      q_k = W_k / N_k: u |q_k|;  v_mix: the two list-order sums over the n_v visited edges, the products and the four outer operations,
        (2 n_v + 8) u A with A = (|vhat| + sum N * sum(p |q|) / sum p) / (sum N + 1) >= |v_mix|;
      e_q = the largest q error (it moves min and max by at most e_q); the span D = max - min by 2 e_q + 2 u D, the floor max(D, 1e-8)
        by as much (max is 1-Lipschitz);  (q - min) / floor: (dq_k + e_q + 2 u |q - min|) / floor_lo + qh dD / floor_lo + 2 u qh;
      sigma = ((c_visit + max N) * c_scale) * qh: C dqh + 3 u C qh;  z = logit + sigma: + 2 u |z|;
      exp(z - max z): the argument off by dz_k + max dz + 2 u |z - max z|, expf within 2 ulp (5 u);  the list-order sum S within the
        largest term error + (n + 2) u;  the division: u.  pi_f32 / pi_64 lies in [(1 - r)(1 - u) / (1 + r_S), (1 + r)(1 + u) / (1 - r_S)].
    Terms below the f32 underflow are covered by an absolute 2^-126."""
    u = 2.0 ** -24
    N = np.asarray(N, np.int64)
    W, P = np.asarray(W, F32).astype(np.float64), np.asarray(P, F32).astype(np.float64)
    logit = np.asarray(logit, F32).astype(np.float64)
    vhat = float(F32(vhat))
    c_visit, c_scale = float(F32(c_visit)), float(F32(c_scale))
    n = len(N)
    vis = N > 0
    nv, sn = int(vis.sum()), int(N.sum())
    qv = W[vis] / N[vis]
    p = np.maximum(P[vis], float(FLT_MIN))
    if sn > 0:
        vm = (vhat + sn * ((p * qv).sum() / p.sum())) / (sn + 1)
        A = (abs(vhat) + sn * (p * np.abs(qv)).sum() / p.sum()) / (sn + 1)
        dvm = (2 * nv + 8) * u * A
    else:
        vm, dvm = vhat, 0.0
    q = np.full(n, vm)
    q[vis] = qv
    dq = np.full(n, dvm)
    dq[vis] = u * np.abs(qv)
    eq = dq.max()
    mn, mx = q.min(), q.max()
    floor = float(F32(1e-8))
    den = max(mx - mn, floor)
    dD = 2 * eq + 2 * u * (mx - mn)
    den_lo = max(den - dD, floor)
    a = q - mn
    qh = a / den
    dqh = (dq + eq + 2 * u * np.abs(a) + qh * dD) / den_lo + 2 * u * qh
    C = (c_visit + float(N.max())) * c_scale
    sig = C * qh
    dsig = C * dqh + 3 * u * C * qh
    z = logit + sig
    fin = np.isfinite(z)
    pi = np.zeros(n)
    bound = np.zeros(n)
    if not fin.any():
        return pi, bound
    dz = np.where(fin, dsig + 2 * u * np.abs(np.where(fin, z, 0.0)), 0.0)
    zm = z[fin].max()
    e = np.where(fin, np.exp(np.where(fin, z - zm, -np.inf)), 0.0)
    pi = e / e.sum()
    arg = dz + dz[fin].max() + 2 * u * np.abs(np.where(fin, z - zm, 0.0))
    with np.errstate(over="ignore", invalid="ignore"):
        r = np.expm1(arg) + 5 * u
        rs = r[fin].max() + (n + 2) * u
        rel = np.where(np.isfinite(r) & (rs < 1), (1 + r) * (1 + u) / (1 - min(rs, 0.5)) - 1, np.inf)
    bound = np.where(fin, pi * rel * (1 + 1e-6) + 2.0 ** -126, 0.0)
    return pi, bound
