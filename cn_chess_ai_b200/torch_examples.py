"""TorchExamples: the self-play example buffer of an AlphaZero-style loop on the device (include/xq.h: xq_examples_*).

Each move, record(search) stores one example per env from its search tree's root: the position and the root edges' visit counts in
sparse form.  When games end, finish(step) (or end_games) stamps each stored position of those games with the result from its side to
move and commits them to a ring.  sample() draws a training batch -- observation planes, the visit-count policy target, the value
target z, the root q and the packed legal mask -- with no host synchronisation.  Calls run on torch's current stream.
"""
from collections import namedtuple

import torch

from ._lib import MASK_WORDS, POLICY_ACTIONS
from .env import BatchedExamples
from .torch_env import _OBS_DTYPES, _view

Sample = namedtuple("Sample", "planes policy value q mask index")

# xq_env_rec piece codes of the Generals (StepResult.captured)
RED_GENERAL, BLACK_GENERAL = 1, 8


class TorchExamples:
    """the example buffer of the envs of `tsearch_or_tenv` (a TorchSearch or a TorchEnv): `capacity` committed examples, and up to
    max_game_examples staged examples per env for the game in progress"""

    def __init__(self, tsearch_or_tenv, capacity, max_game_examples=256):
        self.tenv = getattr(tsearch_or_tenv, "tenv", tsearch_or_tenv)
        self.n = self.tenv.n
        self.device = self.tenv.device
        self.examples = BatchedExamples(self.tenv.env, capacity, max_game_examples)
        self.capacity = self.examples.capacity
        self.max_game_examples = self.examples.max_game_examples

    def close(self):
        self.examples.close()

    def _flags(self, t, name):
        """a bool / uint8 [n] tensor as the uint8 flags the library reads"""
        self.tenv._check(t, name, [torch.bool, torch.uint8], (self.n,))
        return t.view(torch.uint8) if t.dtype == torch.bool else t

    def record(self, search, mask=None):
        """one example of every root of `search` (a TorchSearch on the same envs), or of the envs where mask (bool / uint8 [n]) is set.
        Call it after the search and before the step: a root that is no longer its env's board is skipped and counted as stale."""
        m = None if mask is None else self._flags(mask, "mask")
        self.tenv._enter()
        self.examples.record_device(search.search, None if m is None else m.data_ptr())

    def end_games(self, ended, result_red):
        """commit the staged examples of the envs where ended (bool / uint8 [n]) is set; result_red f32 [n] is each game's result from
        Red's side (NaN -> 0, clamped to [-1, 1]); an example's z is the result from its side to move"""
        e = self._flags(ended, "ended")
        self.tenv._check(result_red, "result_red", [torch.float32], (self.n,))
        self.tenv._enter()
        self.examples.end_games_device(e.data_ptr(), result_red.data_ptr())

    @staticmethod
    def step_results(step, cap_value=0.0):
        """(ended bool [n], result f32 [n] from Red's side) of a TorchEnv.step StepResult: +1 when Black's General was captured, -1 when
        Red's was, cap_value otherwise (the move cap; StepResult.winner is not read, it is Red at the cap whatever the board)"""
        cap = step.captured.to(torch.int32)
        r = torch.full(cap.shape, float(cap_value), dtype=torch.float32, device=cap.device)
        r = torch.where(cap == BLACK_GENERAL, torch.ones_like(r), r)
        r = torch.where(cap == RED_GENERAL, -torch.ones_like(r), r)
        return step.done != 0, r

    def finish(self, step, cap_value=0.0):
        """end_games for the games a TorchEnv.step ended (call it after the step, with the StepResult); returns the ended mask.  Games
        that end without a step reporting done (a side without a legal action) go through end_games."""
        ended, result = self.step_results(step, cap_value)
        self.end_games(ended.contiguous(), result)
        return ended

    def discard(self, mask=None):
        """drop the staged examples of the envs where mask is set (None = all), e.g. after TorchEnv.env.reset / set_boards"""
        m = None if mask is None else self._flags(mask, "mask")
        self.tenv._enter()
        self.examples.discard_device(None if m is None else m.data_ptr())

    def sample(self, batch, seed, counter, view="side", dtype=torch.bfloat16, want_mask=False):
        """Sample of tensors: planes [batch, 14, 10, 9] (dtype), policy f32 [batch, 8100] (visit fractions in the frame of `view`),
        value f32 [batch] (z), q f32 [batch], mask int32 [batch, 254] of packed legal-mask words (want_mask) or None, index int64 [batch]
        (ring slots, -1 while the ring is empty).  Slot i = (xq_rng(seed, i, counter) >> 1) % size."""
        if dtype not in _OBS_DTYPES:
            raise ValueError(f"dtype must be one of {list(_OBS_DTYPES)}")
        v = _view(view)
        batch = int(batch)
        if batch <= 0:
            raise ValueError(f"batch must be > 0, not {batch}")
        self.tenv._enter()
        dev = self.device
        planes = torch.empty((batch, 14, 10, 9), dtype=dtype, device=dev)
        policy = torch.empty((batch, POLICY_ACTIONS), dtype=torch.float32, device=dev)
        value, q = (torch.empty(batch, dtype=torch.float32, device=dev) for _ in range(2))
        mask = torch.empty((batch, MASK_WORDS), dtype=torch.int32, device=dev) if want_mask else None
        index = torch.empty(batch, dtype=torch.int64, device=dev)
        self.examples.sample_device(batch, seed, counter, v, planes.data_ptr(), _OBS_DTYPES[dtype], policy.data_ptr(), value.data_ptr(),
                                    q.data_ptr(), None if mask is None else mask.data_ptr(), index.data_ptr())
        return Sample(planes, policy, value, q, mask, index)

    def info(self):
        """synchronous: dict of size, capacity, total_committed, pending (staged examples), dropped, stale"""
        self.tenv._enter()
        return self.examples.info()

    def __len__(self):
        return self.info()["size"]

    def get(self, first=0, n=None):
        """synchronous read-back of ring slots [first, first + n) as a numpy EXAMPLE_DTYPE array"""
        self.tenv._enter()
        return self.examples.get(first, n)
