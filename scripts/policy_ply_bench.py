"""Times the external-policy interface (xq_env_observe_device, xq_env_legal_mask_device, xq_env_policy_step_device) against the
composed alternative a PyTorch policy needs without it: ordered lists (xq_env_legal_moves_device) -> dense mask (scatter) -> masked_fill
-> log_softmax -> multinomial -> index conversion to xq_action -> xq_env_step_device.

CUDA events around K back-to-back calls (after W warm-up calls) on boards in mid-game (a random-policy rollout first); the score
tensors are [n, 8100] f32, larger than L2 at 65,536 envs.  Prints one JSON object (and writes it to --out): per operation us per ply,
env steps/s, the algorithmic bytes per env and the fraction of the measured copy peak of one B200 (6,458.7 GB/s, BASELINE.md) those
bytes reach.  Also checks that fused GREEDY and the composed argmax pick the same actions on tie-free scores.

    python scripts/policy_ply_bench.py --sizes 4096 65536 --iters 50 --out policy_ply_bench.json
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import cn_chess_ai_b200 as xq  # noqa: E402

COPY_PEAK = 6458.7e9


class _Dev:
    """a device buffer owned by the library, seen by torch through __cuda_array_interface__"""

    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"data": (ptr, False), "shape": shape, "typestr": typestr, "version": 2}


def gpu_info(dev):
    name = torch.cuda.get_device_name(dev)
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:      # the timing does not depend on it; the record says it is missing
        out = f"unavailable ({e})"
    return {"device": name, "power_limit_and_max_sm_clock": out}


def timed(fn, iters, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / iters      # us per call


def run_size(n, iters, warmup, seed=7):
    L = xq.lib()
    dev = torch.device("cuda", 0)
    te = xq.TorchEnv(n, seed=seed)
    te.env.rollout_random(24)                    # mid-game boards
    te._enter()
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    scores = torch.randn((n, 8100), generator=g, device=dev)        # tie-free
    counts_p, lists_p = C.c_void_p(), C.c_void_p()
    L.xq_env_legal_moves_device(te.env.handle, C.byref(counts_p), C.byref(lists_p))
    counts = torch.as_tensor(_Dev(counts_p.value, (n,), "|u1"), device=dev)
    lists = torch.as_tensor(_Dev(lists_p.value, (n, 128), "<i2"), device=dev)
    mean_legal = float(counts.float().mean())

    res = {"envs": n, "mean_legal": mean_legal, "ops": {}}

    def put(name, us, bytes_per_env):
        res["ops"][name] = {"us_per_ply": round(us, 2), "env_steps_per_s": n / us * 1e6, "bytes_per_env": round(bytes_per_env, 1),
                            "frac_copy_peak": bytes_per_env * n / (us * 1e-6) / COPY_PEAK}

    planes = {dt: torch.empty((n, 14, 10, 9), dtype=dt, device=dev) for dt in (torch.float32, torch.bfloat16, torch.uint8)}
    aux = torch.empty((n, 4), dtype=torch.int32, device=dev)
    for dt, code, sz in ((torch.float32, 0, 4), (torch.bfloat16, 1, 2), (torch.uint8, 2, 1)):
        us = timed(lambda: te.env.observe_device(planes[dt].data_ptr(), code, 1, aux.data_ptr()), iters, warmup)
        put(f"observe_{str(dt).split('.')[-1]}", us, 64 + 1260 * sz + 16)
    dense = torch.empty((n, 8100), dtype=torch.bool, device=dev)
    packed = torch.empty((n, 254), dtype=torch.int32, device=dev)
    put("mask_dense", timed(lambda: te.env.legal_mask_device(dense.data_ptr(), False, 1), iters, warmup), 64 + 8100)
    put("mask_packed", timed(lambda: te.env.legal_mask_device(packed.data_ptr(), True, 1), iters, warmup), 64 + 1016)

    # fused GREEDY vs the composed argmax on the same boards, before any step
    L.xq_env_legal_moves_device(te.env.handle, None, None)
    a = lists.int() & 0xFFFF
    idx = torch.where(a != 0xFFFF, (a >> 7) * 90 + (a & 127), 8100).long()
    m = torch.zeros((n, 8101), dtype=torch.bool, device=dev).scatter_(1, idx, True)[:, :8100]
    comp_greedy = scores.masked_fill(~m, float("-inf")).argmax(1)
    fused_greedy = te.step(scores, pick="greedy", view="absolute", auto_reset=False).actions     # applies the ply (boards move on)
    has = m.any(1)
    agree = bool((fused_greedy[has] == comp_greedy[has]).all())
    res["greedy_matches_composed_argmax"] = agree

    act = torch.empty(n, dtype=torch.int64, device=dev)
    logp = torch.empty(n, dtype=torch.float32, device=dev)
    rew = torch.empty(n, dtype=torch.int32, device=dev)
    u8 = [torch.empty(n, dtype=torch.uint8, device=dev) for _ in range(4)]
    outs = [rew.data_ptr()] + [t.data_ptr() for t in u8]
    step_bytes = 64 + 64 + 32 * mean_legal + 20

    def fused(pick, lp):
        te.env.policy_step_device(scores.data_ptr(), 0, pick, 1.0, 1, True, act.data_ptr(), logp.data_ptr() if lp else None, *outs)
    put("step_greedy", timed(lambda: fused(0, False), iters, warmup), step_bytes)
    put("step_greedy_logp", timed(lambda: fused(0, True), iters, warmup), step_bytes)
    put("step_sample", timed(lambda: fused(1, True), iters, warmup), step_bytes)

    # GIVEN: a second handle in lockstep (same seed, same boards) samples the actions; GIVEN time = window - the sampling alone
    tb = xq.TorchEnv(n, seed=seed)
    tb.env.set_boards(te.env.get_boards())
    act_b = torch.empty(n, dtype=torch.int64, device=dev)

    def sample_b():
        tb.env.policy_step_device(scores.data_ptr(), 0, 1, 1.0, 1, True, act_b.data_ptr(), None, None, None, None, None, None)

    def pair():
        sample_b()
        te.env.policy_step_device(scores.data_ptr(), 0, 2, 1.0, 1, True, act_b.data_ptr(), logp.data_ptr(), *outs)
    t_pair = timed(pair, iters, warmup)
    t_b = timed(sample_b, iters, warmup)
    put("step_given_logp", t_pair - t_b, step_bytes)
    res["ops"]["step_given_logp"]["note"] = "pair (SAMPLE on a lockstep handle + GIVEN) minus SAMPLE alone"

    # the composed alternative
    xa = torch.empty(n, dtype=torch.int16, device=dev)

    def composed():
        L.xq_env_legal_moves_device(te.env.handle, None, None)
        a = lists.int() & 0xFFFF
        idx = torch.where(a != 0xFFFF, (a >> 7) * 90 + (a & 127), 8100).long()
        mk = torch.zeros((n, 8101), dtype=torch.bool, device=dev).scatter_(1, idx, True)[:, :8100]
        mk[:, 0] |= ~mk.any(1)                   # multinomial needs one non-zero weight per row (an empty list plays nothing below)
        lp = torch.log_softmax(scores.masked_fill(~mk, float("-inf")), 1)
        k = torch.multinomial(lp.exp(), 1).squeeze(1)
        lp.gather(1, k[:, None])
        xa.copy_(torch.where(counts > 0, (k // 90) << 7 | (k % 90), 0xFFFF).to(torch.int16))
        L.xq_env_step_device(te.env.handle, C.c_void_p(xa.data_ptr()), 1, None, None, None, None, None)
    put("composed_sample", timed(composed, max(iters // 2, 5), warmup), 64 + 256 + 1 + 8100 * 4 * 3 + 8100 * 2 + 64 + 20)
    res["ops"]["composed_sample"]["note"] = "bytes: lists + mask + scores read, masked logits and log-probs written and read (lower bound)"
    tb.close()
    te.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[4096, 65536])
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("policy_ply_bench: no GPU")
    out = {"gpu": gpu_info(0), "copy_peak_Bps": COPY_PEAK, "sizes": [run_size(n, args.iters, args.warmup) for n in args.sizes]}
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
