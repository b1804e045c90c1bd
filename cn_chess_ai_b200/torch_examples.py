"""TorchExamples: the self-play example buffer of an AlphaZero-style loop on the device (include/xq.h: xq_examples_*).

Each move, record(search) stores one example per env from its search tree's root: the position and the root edges' visit counts in
sparse form.  When games end, finish(step) (or end_games) stamps each stored position of those games with the result from its side to
move and commits them to a ring.  sample() draws a training batch -- observation planes, the visit-count policy target, the value
target z, the root q and the packed legal mask -- with no host synchronisation.  reanalyse() searches stored positions again with the
current network and rewrites their policy targets and q in place (load, a search, refresh).  Calls run on torch's current stream.
"""
from collections import namedtuple

import torch

from ._lib import COMPACT_ACTIONS, MASK_WORDS, POLICY_ACTIONS
from .env import BatchedExamples
from .torch_env import _OBS_DTYPES, _view

Sample = namedtuple("Sample", "planes policy value q mask index")
CompactSample = namedtuple("CompactSample", "planes actions policy counts value q index")

# xq_env_rec piece codes of the Generals (StepResult.captured)
RED_GENERAL, BLACK_GENERAL = 1, 8

# status of a refreshed row (include/xq.h: XQ_REFRESH*), checked in this order: the slot is rewritten; the index is < 0 or >= len(); a
# smaller row has the same index (only the smallest writes); the slot's record is no longer the root's (the ring wrapped over it); the
# root has no edge with a visit or a weight
REFRESHED, NO_SLOT, DUPLICATE, STALE, UNSEARCHED = 0, 1, 2, 3, 4


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

    def record_gumbel(self, gumbel, mask=None):
        """record() after a Gumbel search (a TorchGumbel on the same envs): the stored visits are the integer weights
        round(pi'_k * 2^24) of the improved policy, so sample() gives pi' (within about 2^-24) as the policy target"""
        m = None if mask is None else self._flags(mask, "mask")
        self.tenv._enter()
        self.examples.record_gumbel_device(gumbel.gumbel, None if m is None else m.data_ptr())

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

    def sample(self, batch, seed, counter, view="side", dtype=torch.bfloat16, want_mask=False, compact=False):
        """Sample of tensors: planes [batch, 14, 10, 9] (dtype), policy f32 [batch, 8100] (visit fractions in the frame of `view`),
        value f32 [batch] (z), q f32 [batch], mask int32 [batch, 254] of packed legal-mask words (want_mask) or None, index int64 [batch]
        (ring slots, -1 while the ring is empty).  Slot i = (xq_rng(seed, i, counter) >> 1) % size.
        compact=True: the same rows as a CompactSample -- planes, actions int32 [batch, 128] (the root's edges as policy indices in the
        frame of `view`, list order, -1 past them), policy f32 [batch, 128] (the visit fraction of edge k), counts uint8 [batch] (edges),
        value, q, index."""
        if dtype not in _OBS_DTYPES:
            raise ValueError(f"dtype must be one of {list(_OBS_DTYPES)}")
        v = _view(view)
        batch = int(batch)
        if batch <= 0:
            raise ValueError(f"batch must be > 0, not {batch}")
        if compact and want_mask:
            raise ValueError("want_mask is for the dense policy row: a compact sample lists the actions instead")
        self.tenv._enter()
        dev = self.device
        planes = torch.empty((batch, 14, 10, 9), dtype=dtype, device=dev)
        if compact:
            actions = torch.empty((batch, COMPACT_ACTIONS), dtype=torch.int32, device=dev)
            policy = torch.empty((batch, COMPACT_ACTIONS), dtype=torch.float32, device=dev)
            counts = torch.empty(batch, dtype=torch.uint8, device=dev)
            value, q = (torch.empty(batch, dtype=torch.float32, device=dev) for _ in range(2))
            index = torch.empty(batch, dtype=torch.int64, device=dev)
            self.examples.sample_compact_device(batch, seed, counter, v, planes.data_ptr(), _OBS_DTYPES[dtype], actions.data_ptr(),
                                                policy.data_ptr(), counts.data_ptr(), value.data_ptr(), q.data_ptr(), index.data_ptr())
            return CompactSample(planes, actions, policy, counts, value, q, index)
        policy = torch.empty((batch, POLICY_ACTIONS), dtype=torch.float32, device=dev)
        value, q = (torch.empty(batch, dtype=torch.float32, device=dev) for _ in range(2))
        mask = torch.empty((batch, MASK_WORDS), dtype=torch.int32, device=dev) if want_mask else None
        index = torch.empty(batch, dtype=torch.int64, device=dev)
        self.examples.sample_device(batch, seed, counter, v, planes.data_ptr(), _OBS_DTYPES[dtype], policy.data_ptr(), value.data_ptr(),
                                    q.data_ptr(), None if mask is None else mask.data_ptr(), index.data_ptr())
        return Sample(planes, policy, value, q, mask, index)

    def load(self, tenv, index):
        """env e of `tenv` (any TorchEnv on the buffer's device) gets the record of ring slot index[e] (int64 [tenv.n], e.g. sample().index
        or a torch.arange sweep), all 64 bytes, so that a search reset on tenv has exactly the stored position as its root.  Rows with
        an index < 0 or >= len() keep their board.  As after tenv.env.set_boards, staged examples of a buffer on tenv are stale."""
        tenv._check(index, "index", [torch.int64], (tenv.n,))
        self.tenv._enter()
        tenv._enter()
        self.examples.load_device(tenv.env, index.data_ptr())

    def refresh(self, search, index):
        """tree t of `search` (a TorchSearch on any TorchEnv of the device, after its simulations) rewrites n_edges, action, visits,
        total_visits and q of ring slot index[t] (int64 [search.n]) as record() would store them from that tree; rec, env, game, ply and z
        stay.  Returns the status uint8 [search.n] of each row (REFRESHED .. UNSEARCHED)."""
        return self._refresh(search.tenv, search.n, index, lambda i, st: self.examples.refresh_device(search.search, i, st))

    def refresh_gumbel(self, gumbel, index):
        """refresh() after a Gumbel search (a begun TorchGumbel): visits are the weights of record_gumbel()"""
        return self._refresh(gumbel.tenv, gumbel.n, index, lambda i, st: self.examples.refresh_gumbel_device(gumbel.gumbel, i, st))

    def _refresh(self, tenv, n, index, call):
        tenv._check(index, "index", [torch.int64], (n,))
        status = torch.empty(n, dtype=torch.uint8, device=self.device)
        self.tenv._enter()
        tenv._enter()
        call(index.data_ptr(), status.data_ptr())
        return status

    def reanalyse(self, runner, evaluate, index, n_simulations, **run_kwargs):
        """Reanalyse: search the positions of ring slots index (int64 [runner.n]) again with `evaluate` and rewrite their policy targets
        and q.  load(runner.tenv, index), then runner.run(evaluate, n_simulations, reset=True, **run_kwargs) (a TorchSearch or a
        TorchGumbel; compact=True and leaves=L pass through; no Dirichlet noise unless run_kwargs ask for it), then refresh() (or
        refresh_gumbel()).  Returns the statuses."""
        from .torch_search import TorchGumbel
        self.load(runner.tenv, index)
        runner.run(evaluate, n_simulations, reset=True, **run_kwargs)
        return self.refresh_gumbel(runner, index) if isinstance(runner, TorchGumbel) else self.refresh(runner, index)

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
