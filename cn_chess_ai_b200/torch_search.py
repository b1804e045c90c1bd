"""TorchSearch: batched PUCT tree search (one tree per env) for a policy/value network written in PyTorch, on the device
(include/xq.h: xq_search_*).

Each simulation selects one leaf per tree (or, with select_leaves, several per tree with virtual loss), observes all leaves at once, calls
the network once on them and hands its scores and values back; selection, child creation, expansion and backup run in the library's
kernels on torch's current stream.  Actions and visit counts
use the policy indices from * 90 + to of TorchEnv, in the frame of `view`.
"""
from collections import namedtuple

import torch

from ._lib import POLICY_ACTIONS, SEARCH_MAX_EDGES
from .env import BatchedGumbel, BatchedSearch
from .torch_env import _OBS_DTYPES, _SCORE_DTYPES, StepResult, _view

SelectResult = namedtuple("SelectResult", "status winner reward depth")
RootResult = namedtuple("RootResult", "visits q best")

# leaf status (xq_search_select_device; DUPLICATE only from xq_search_select_leaves_device)
NEEDS_EVALUATION, GENERAL_CAPTURED, MOVE_CAP, NO_LEGAL_ACTION, DUPLICATE = 0, 1, 2, 3, 4


class TorchSearch:
    """max_simulations simulations per reset on the envs of `tenv` (a TorchEnv); the roots are the envs' boards at reset().  max_leaves:
    the most leaves per tree one select_leaves() call may take (1 .. 32)"""

    def __init__(self, tenv, max_simulations, max_leaves=1):
        self.tenv = tenv
        self.n = tenv.n
        self.device = tenv.device
        self.search = BatchedSearch(tenv.env, max_simulations, max_leaves)
        self.max_simulations = self.search.max_simulations
        self.max_leaves = self.search.max_leaves
        self._rows = self.n        # leaf rows of the last selection: n * leaves
        self._kept = None          # kept int32 [n] of the last advance(); None after reset(): every root was rebuilt

    def close(self):
        self.search.close()

    def reset(self):
        self.tenv._enter()
        self.search.reset()
        self._kept = None

    def advance(self, min_free, root_noise=None, noise_eps=0.25, view="side"):
        """instead of reset() after a move: every tree is re-rooted at its env's current board, keeping the subtree (and its statistics)
        of the child that was played, or rebuilt as reset() builds it when nothing matches (a game that ended and was reset) or the
        subtree has more than max_simulations + 1 - min_free nodes.  Exactly min_free simulations are allowed afterwards.  root_noise
        f32 [n, 8100] (frame of `view`): mixed into the priors of every kept, expanded root.  Returns kept int32 [n]: nodes carried over,
        0 for a rebuilt tree."""
        v = _view(view)
        if root_noise is not None:
            self.tenv._check(root_noise, "root_noise", [torch.float32], (self.n, POLICY_ACTIONS))
        self.tenv._enter()
        kept = torch.empty(self.n, dtype=torch.int32, device=self.device)
        self.search.advance_device(min_free, None if root_noise is None else root_noise.data_ptr(), noise_eps, v, kept.data_ptr())
        self._kept = kept
        return kept

    def select(self, c_puct=1.5, fpu=0.0):
        """one leaf per tree: SelectResult of tensors [n]: status / winner uint8, reward / depth int32"""
        self.tenv._enter()
        sel = self._select_outputs(self.n)
        self.search.select_device(c_puct, fpu, *(t.data_ptr() for t in sel))
        self._rows = self.n
        return sel

    def select_leaves(self, leaves, c_puct=1.5, fpu=0.0, virtual_loss=1.0):
        """`leaves` leaves per tree in one call, descents in order with virtual loss (include/xq.h): SelectResult of tensors [n, leaves];
        status DUPLICATE (4) marks a slot that ended at the open leaf of an earlier slot.  leaves(), observe() and expand_backup() then
        take or return n * leaves rows, slot k of tree t at row t * leaves + k.  Spends `leaves` of the search's simulations."""
        self.tenv._enter()
        sel = self._select_outputs((self.n, int(leaves)))
        self.search.select_leaves_device(leaves, c_puct, fpu, virtual_loss, *(t.data_ptr() for t in sel))
        self._rows = self.n * int(leaves)
        return sel

    def _select_outputs(self, shape):
        """the SelectResult tensors a select call fills: status / winner uint8, reward / depth int32 of `shape`"""
        return SelectResult(*(torch.empty(shape, dtype=dt, device=self.device) for dt in (torch.uint8, torch.uint8, torch.int32, torch.int32)))

    def leaves(self):
        """the leaf records of the last selection as a uint8 [rows, 64] tensor aliasing the library's buffer (xq_env_rec each, rows = n
        after select(), n * leaves after select_leaves(); valid until the next select: clone() to keep them)"""
        ptr = self.search.leaves_device()
        n = self._rows

        class _Leaves:
            __cuda_array_interface__ = {"shape": (n, 64), "typestr": "|u1", "data": (ptr, False), "version": 3, "strides": None}

        return torch.as_tensor(_Leaves(), device=self.device)

    def observe(self, dtype=torch.bfloat16, view="side"):
        """the leaves as TorchEnv.observe shows envs: (planes [rows, 14, 10, 9], aux int32 [rows, 4]), rows as in leaves()"""
        if dtype not in _OBS_DTYPES:
            raise ValueError(f"dtype must be one of {list(_OBS_DTYPES)}")
        v = _view(view)
        self.tenv._enter()
        planes = torch.empty((self._rows, 14, 10, 9), dtype=dtype, device=self.device)
        aux = torch.empty((self._rows, 4), dtype=torch.int32, device=self.device)
        self.search.observe_leaves_device(planes.data_ptr(), _OBS_DTYPES[dtype], v, aux.data_ptr())
        return planes, aux

    def expand_backup(self, scores, values, temperature=1.0, root_noise=None, noise_eps=0.25, view="side"):
        """scores [rows, 8100] (f32 / bf16, frame of `view`) expand the leaves that need evaluation; values f32 [rows] (from each leaf's
        side to move) are backed up for every leaf but duplicates (rows as in leaves()).  root_noise f32 [n, 8100]: mixed into the
        root's priors when the root is expanded."""
        v = _view(view)
        self.tenv._check(scores, "scores", list(_SCORE_DTYPES), (self._rows, POLICY_ACTIONS))
        self.tenv._check(values, "values", [torch.float32], (self._rows,))
        if root_noise is not None:
            self.tenv._check(root_noise, "root_noise", [torch.float32], (self.n, POLICY_ACTIONS))
        self.tenv._enter()
        self.search.expand_backup_device(scores.data_ptr(), _SCORE_DTYPES[scores.dtype], temperature, v, values.data_ptr(),
                                         None if root_noise is None else root_noise.data_ptr(), noise_eps)

    def root(self, view="side"):
        """RootResult: visits int32 [n, 8100] (frame of `view`), q f32 [n] (NaN without a visited edge), best int64 [n] (the most-visited
        root action, -1 without a visited edge: the input of TorchEnv.step(actions=best, pick="given"))"""
        v = _view(view)
        self.tenv._enter()
        visits = torch.empty((self.n, POLICY_ACTIONS), dtype=torch.int32, device=self.device)
        q = torch.empty(self.n, dtype=torch.float32, device=self.device)
        best = torch.empty(self.n, dtype=torch.int64, device=self.device)
        self.search.root_device(v, visits.data_ptr(), q.data_ptr(), best.data_ptr())
        return RootResult(visits, q, best)

    def play(self, temperature=1.0, sample_plies=30, view="side", auto_reset=True):
        """one move per env from its root's visit counts, played on the env: sampled with probability N^(1 / temperature) while the root's
        move_count < sample_plies, the most-visited edge afterwards or at temperature 0.  A root that is not its env's board or has no
        visited edge plays nothing (action -1, valid 0).  Returns a TorchEnv.step StepResult (logp None): actions int64 (frame of `view`),
        reward i32, done / winner / captured / valid uint8 -- the input of TorchExamples.finish.  The trees are not changed: advance()
        re-roots them at the played moves."""
        v = _view(view)
        self.tenv._enter()
        res = self._step_outputs()
        self.search.play_device(temperature, sample_plies, v, auto_reset, *(t.data_ptr() for t in res if t is not None))
        return res

    def _step_outputs(self):
        """the StepResult tensors [n] a play call fills: actions int64, logp None, reward int32, done / winner / captured / valid uint8"""
        empty = lambda dt: torch.empty(self.n, dtype=dt, device=self.device)      # noqa: E731
        return StepResult(empty(torch.int64), None, empty(torch.int32), *(empty(torch.uint8) for _ in range(4)))

    def root_noise(self, alpha, eps=0.25, seed=0, mask=None, want_noise=False):
        """Dirichlet(alpha) noise drawn by the library over the edges of every expanded root (or of the envs where mask, bool / uint8 [n],
        is set) and mixed into its priors: P <- (1 - eps) P + eps eta.  The draw depends on the seed, the global env id and the root's
        ply counter only.  Returns eta f32 [n, 128] in the root's edge order (0 past its edges and for trees left alone) with want_noise,
        else None."""
        m = None
        if mask is not None:
            self.tenv._check(mask, "mask", [torch.bool, torch.uint8], (self.n,))
            m = mask.view(torch.uint8) if mask.dtype == torch.bool else mask
        self.tenv._enter()
        out = torch.empty((self.n, SEARCH_MAX_EDGES), dtype=torch.float32, device=self.device) if want_noise else None
        self.search.root_noise_device(alpha, eps, seed, None if m is None else m.data_ptr(), None if out is None else out.data_ptr())
        return out

    @staticmethod
    def outcome_values(status, winner, aux, cap_value=0.0):
        """a default value of terminal leaves, from the leaf's side to move (aux[:, 0], absolute colour): +1 / -1 when a General was
        captured and the side to move is / is not the winner, cap_value at the move cap, -1 without a legal action, 0 elsewhere
        (duplicates included)"""
        player = aux[:, 0].to(torch.int32)
        won = torch.where(winner.to(torch.int32) == player, 1.0, -1.0)
        v = torch.zeros(status.shape, dtype=torch.float32, device=status.device)
        v = torch.where(status == GENERAL_CAPTURED, won, v)
        v = torch.where(status == MOVE_CAP, torch.full_like(v, float(cap_value)), v)
        return torch.where(status == NO_LEGAL_ACTION, torch.full_like(v, -1.0), v)

    def run(self, evaluate, n_simulations, c_puct=1.5, fpu=0.0, temperature=1.0, root_noise=None, noise_eps=0.25, view="side",
            obs_dtype=torch.bfloat16, cap_value=0.0, reset=True, dirichlet_alpha=None, dirichlet_eps=0.25, noise_seed=0, leaves=1,
            virtual_loss=1.0):
        """reset + n_simulations simulations: evaluate(planes) -> (scores [rows, 8100], values [rows]) is called once per selection on
        its leaves; at terminal leaves outcome_values replaces the network's value.  reset=False continues from the current trees (after
        advance(), or to add simulations to this move's search).  dirichlet_alpha: root_noise(dirichlet_alpha, dirichlet_eps, noise_seed)
        once per root and move -- before the first simulation on the roots the last advance() kept, after it on the roots reset() or
        advance() rebuilt (expanded by the first simulation).  leaves > 1: after the first simulation (one leaf per tree, which expands
        rebuilt roots) the rest go in select_leaves(leaves, virtual_loss=virtual_loss) calls, the last one smaller, so evaluate sees
        n * leaves planes; n_simulations counts the selected slots.  Returns root(view)."""
        if reset:
            self.reset()
        kept = None if self._kept is None else self._kept > 0
        if dirichlet_alpha is not None and kept is not None:
            self.root_noise(dirichlet_alpha, dirichlet_eps, noise_seed, mask=kept)
        i = 0
        while i < n_simulations:
            if i == 1 and dirichlet_alpha is not None:
                self.root_noise(dirichlet_alpha, dirichlet_eps, noise_seed, mask=None if kept is None else ~kept)
            k = 1 if i == 0 else min(leaves, n_simulations - i)
            sel = self.select(c_puct, fpu) if k == 1 else self.select_leaves(k, c_puct, fpu, virtual_loss)
            self._simulate(sel, evaluate, temperature, root_noise, noise_eps, view, obs_dtype, cap_value)
            i += k
        return self.root(view)

    def _simulate(self, sel, evaluate, temperature, root_noise, noise_eps, view, obs_dtype, cap_value):
        """the rest of a simulation after the selection `sel`: its leaves observed and evaluated once, outcome_values at terminal leaves,
        expand_backup"""
        status, winner = sel.status.reshape(-1), sel.winner.reshape(-1)
        planes, aux = self.observe(obs_dtype, view)
        scores, values = evaluate(planes)
        values = values.reshape(self._rows).to(torch.float32).contiguous()
        values = torch.where(status != NEEDS_EVALUATION, self.outcome_values(status, winner, aux, cap_value), values)
        self.expand_backup(scores.contiguous(), values, temperature, root_noise, noise_eps, view)


GumbelRootResult = namedtuple("GumbelRootResult", "policy action")


class TorchGumbel:
    """Gumbel root search (Danihelka et al., ICLR 2022; include/xq.h: xq_gumbel_*) on a TorchSearch: each move begin() samples up to
    max_considered (1 .. 128) root actions per tree without replacement (Gumbel-top-k), select() splits the move's simulations among them
    by Sequential Halving, root() gives the improved policy pi' = softmax(logits + sigma(completed Q)) -- the policy target -- and the
    action to play, play() plays it.  Below the root, selection is the search's PUCT (with virtual loss for several leaves)."""

    def __init__(self, search, max_considered=16):
        self.tsearch = search
        self.tenv = search.tenv
        self.n = search.n
        self.device = search.device
        self.gumbel = BatchedGumbel(search.search, max_considered)
        self.max_considered = self.gumbel.max_considered

    def close(self):
        self.gumbel.close()

    def begin(self, scores, values, n_simulations, seed=0, temperature=1.0, c_visit=50.0, c_scale=0.1, view="side"):
        """after the search's reset() / advance(): scores [n, 8100] (f32 / bf16, frame of `view`) and values f32 [n] of the network on the
        roots (TorchEnv.observe).  Unexpanded roots are expanded and backed up from them, as a first simulation would; then every tree
        draws its Gumbels from (seed, env id, root ply counter), picks its considered actions and keeps the root value for the completed
        Q.  n_simulations: the selected slots of this move."""
        v = _view(view)
        self.tenv._check(scores, "scores", list(_SCORE_DTYPES), (self.n, POLICY_ACTIONS))
        self.tenv._check(values, "values", [torch.float32], (self.n,))
        self.tenv._enter()
        self.gumbel.begin_device(scores.data_ptr(), _SCORE_DTYPES[scores.dtype], temperature, v, values.data_ptr(), n_simulations, seed,
                                 c_visit, c_scale)

    def select(self, leaves=1, c_puct=1.5, fpu=0.0, virtual_loss=1.0):
        """TorchSearch.select_leaves with the Gumbel root rule: SelectResult of tensors [n, leaves]; the search's leaves(), observe() and
        expand_backup() follow as after select_leaves"""
        ts = self.tsearch
        self.tenv._enter()
        sel = ts._select_outputs((self.n, int(leaves)))
        self.gumbel.select_device(leaves, c_puct, fpu, virtual_loss, *(t.data_ptr() for t in sel))
        ts._rows = self.n * int(leaves)
        return sel

    def root(self, view="side"):
        """GumbelRootResult: policy f32 [n, 8100] (pi' in the frame of `view`, zero rows for roots without edges), action int64 [n] (the
        considered action with the most visits this move, -1 without one: the input of TorchEnv.step(actions=action, pick="given"))"""
        v = _view(view)
        self.tenv._enter()
        policy = torch.empty((self.n, POLICY_ACTIONS), dtype=torch.float32, device=self.device)
        action = torch.empty(self.n, dtype=torch.int64, device=self.device)
        self.gumbel.root_device(v, policy.data_ptr(), action.data_ptr())
        return GumbelRootResult(policy, action)

    def play(self, view="side", auto_reset=True):
        """root().action played on every env, as TorchSearch.play steps (a stale root or no action plays nothing): StepResult"""
        v = _view(view)
        self.tenv._enter()
        res = self.tsearch._step_outputs()
        self.gumbel.play_device(v, auto_reset, *(t.data_ptr() for t in res if t is not None))
        return res

    def run(self, evaluate, n_simulations, seed=0, c_puct=1.5, fpu=0.0, temperature=1.0, c_visit=50.0, c_scale=0.1, view="side",
            obs_dtype=torch.bfloat16, cap_value=0.0, leaves=1, virtual_loss=1.0, reset=True):
        """one move's Gumbel search: reset() (reset=False: continue from advance()), evaluate(planes) -> (scores, values) once on the env
        boards (TorchEnv.observe) for begin(), then n_simulations selections in select(leaves) calls, the last one smaller, each
        evaluated once with outcome_values at terminal leaves as TorchSearch.run does.  Returns root(view)."""
        ts = self.tsearch
        if reset:
            ts.reset()
        planes, _ = self.tenv.observe(obs_dtype, view)
        scores, values = evaluate(planes)
        self.begin(scores.contiguous(), values.reshape(self.n).to(torch.float32).contiguous(), n_simulations, seed, temperature, c_visit,
                   c_scale, view)
        i = 0
        while i < n_simulations:
            k = min(leaves, n_simulations - i)
            ts._simulate(self.select(k, c_puct, fpu, virtual_loss), evaluate, temperature, None, 0.0, view, obs_dtype, cap_value)
            i += k
        return self.root(view)
