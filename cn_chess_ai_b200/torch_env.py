"""TorchEnv: the batched environment for a policy written in PyTorch, with observations, legal-action masks and the policy's step
all on the device (include/xq.h: xq_env_observe_device, xq_env_legal_mask_device, xq_env_policy_step_device).

Every call runs on torch.cuda.current_stream(device), allocates its outputs with torch and hands their data_ptr() to the library:
nothing goes through host memory.  Actions are policy indices from * 90 + to (8,100 of them, the reference network's output width);
with view="side" an env with Black to move is seen rotated by 180 degrees with the colours swapped, so that a network always plays
"up the board" with its own pieces in channels 0..6.  A network that scores only the legal actions uses compact rows instead:
legal_actions() lists each board's actions (entry k = list entry k, 128 wide) and step_compact() takes scores in that order.
"""
from collections import namedtuple

import torch

from ._lib import (COMPACT_ACTIONS, DTYPE_BF16, DTYPE_F32, DTYPE_U8, MASK_WORDS, PICK_GIVEN, PICK_GREEDY, PICK_SAMPLE, POLICY_ACTIONS,
                   VIEW_ABSOLUTE, VIEW_SIDE_TO_MOVE)
from .env import BatchedEnv

StepResult = namedtuple("StepResult", "actions logp reward done winner captured valid")

_VIEWS = {"absolute": VIEW_ABSOLUTE, "side": VIEW_SIDE_TO_MOVE}
_PICKS = {"greedy": PICK_GREEDY, "sample": PICK_SAMPLE, "given": PICK_GIVEN}
_OBS_DTYPES = {torch.float32: DTYPE_F32, torch.bfloat16: DTYPE_BF16, torch.uint8: DTYPE_U8}
_SCORE_DTYPES = {torch.float32: DTYPE_F32, torch.bfloat16: DTYPE_BF16}


def _view(view):
    if view not in _VIEWS:
        raise ValueError(f"view must be one of {sorted(_VIEWS)}, not {view!r}")
    return _VIEWS[view]


class TorchEnv:
    """n_envs boards on cuda:<device>; `env` wraps an existing BatchedEnv instead of creating one."""

    def __init__(self, n_envs=None, device=0, seed=0, env_id0=0, env=None):
        self.env = env if env is not None else BatchedEnv(n_envs, device=device, seed=seed, env_id0=env_id0)
        self.n = self.env.n
        self.device = torch.device("cuda", self.env.device)
        self._stream = None

    def close(self):
        self.env.close()

    def _enter(self):
        """the handle follows torch's current stream (set only when it changes: setting it synchronises the previous one)"""
        s = torch.cuda.current_stream(self.device).cuda_stream
        if s != self._stream:
            self.env.set_stream(s)
            self._stream = s

    def _check(self, t, name, dtypes, shape):
        if t.device != self.device or t.dtype not in dtypes or tuple(t.shape) != shape or not t.is_contiguous():
            raise ValueError(f"{name}: want a contiguous {shape} tensor of {[str(d) for d in dtypes]} on {self.device}, "
                             f"got {tuple(t.shape)} {t.dtype} on {t.device}")

    def observe(self, dtype=torch.bfloat16, view="side"):
        """(planes [n, 14, 10, 9] of 0/1 in `dtype`, aux int32 [n, 4] = player, move_count, red_score, black_score)"""
        if dtype not in _OBS_DTYPES:
            raise ValueError(f"dtype must be one of {list(_OBS_DTYPES)}")
        v = _view(view)
        self._enter()
        planes = torch.empty((self.n, 14, 10, 9), dtype=dtype, device=self.device)
        aux = torch.empty((self.n, 4), dtype=torch.int32, device=self.device)
        self.env.observe_device(planes.data_ptr(), _OBS_DTYPES[dtype], v, aux.data_ptr())
        return planes, aux

    def legal_mask(self, packed=False, view="side"):
        """bool [n, 8100] (packed=False) or int32 [n, 254] holding the packed uint32 words (bit i % 32 of word i // 32)"""
        v = _view(view)
        self._enter()
        if packed:
            mask = torch.empty((self.n, MASK_WORDS), dtype=torch.int32, device=self.device)
        else:
            mask = torch.empty((self.n, POLICY_ACTIONS), dtype=torch.bool, device=self.device)
        self.env.legal_mask_device(mask.data_ptr(), packed, v)
        return mask

    def legal_actions(self, view="side"):
        """(actions int32 [n, 128], counts uint8 [n]): entry k of a row is the policy index (frame of `view`) of the env's k-th legal
        action in reference list order, -1 past the count -- the order of a compact score row (step_compact, TorchSearch)"""
        v = _view(view)
        self._enter()
        actions = torch.empty((self.n, COMPACT_ACTIONS), dtype=torch.int32, device=self.device)
        counts = torch.empty(self.n, dtype=torch.uint8, device=self.device)
        self.env.legal_actions_device(actions.data_ptr(), counts.data_ptr(), v)
        return actions, counts

    def step(self, scores=None, actions=None, pick="sample", temperature=1.0, view="side", auto_reset=True):
        """one ply: scores [n, 8100] (f32 / bf16) in the view's frame and/or actions int64 [n] (pick="given").  Returns StepResult of
        tensors: actions int64 (policy indices, -1 = no legal action), logp f32 (NaN without scores), reward i32, done / winner / captured / valid uint8."""
        return self._step(scores, actions, pick, temperature, view, auto_reset, False)

    def step_compact(self, scores=None, actions=None, pick="sample", temperature=1.0, view="side", auto_reset=True):
        """step() with compact scores [n, 128] (f32 / bf16): entry k scores the env's k-th legal action (legal_actions(view)).  actions
        (given and returned) are policy indices in the frame of `view`, as in step(); the same StepResult, bit for bit step()'s with the
        dense row holding the compact entries at their policy indices."""
        return self._step(scores, actions, pick, temperature, view, auto_reset, True)

    def _step(self, scores, actions, pick, temperature, view, auto_reset, compact):
        if pick not in _PICKS:
            raise ValueError(f"pick must be one of {sorted(_PICKS)}, not {pick!r}")
        p, v = _PICKS[pick], _view(view)
        sdt = DTYPE_F32
        if scores is not None:
            self._check(scores, "scores", list(_SCORE_DTYPES), (self.n, COMPACT_ACTIONS if compact else POLICY_ACTIONS))
            sdt = _SCORE_DTYPES[scores.dtype]
        if p == PICK_GIVEN:
            if actions is None:
                raise ValueError('pick="given" needs actions')
            self._check(actions, "actions", [torch.int64], (self.n,))
        else:
            if scores is None:
                raise ValueError(f"pick={pick!r} needs scores")
            actions = torch.empty(self.n, dtype=torch.int64, device=self.device)
        self._enter()
        logp = torch.empty(self.n, dtype=torch.float32, device=self.device)
        reward = torch.empty(self.n, dtype=torch.int32, device=self.device)
        done, winner, captured, valid = (torch.empty(self.n, dtype=torch.uint8, device=self.device) for _ in range(4))
        call = self.env.policy_step_compact_device if compact else self.env.policy_step_device
        call(None if scores is None else scores.data_ptr(), sdt, p, temperature, v, auto_reset, actions.data_ptr(), logp.data_ptr(),
             reward.data_ptr(), done.data_ptr(), winner.data_ptr(), captured.data_ptr(), valid.data_ptr())
        return StepResult(actions, logp, reward, done, winner, captured, valid)
