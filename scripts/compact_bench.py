"""Times the compact score rows (include/xq.h: XQ_COMPACT_ACTIONS) against the dense [rows, 8100] rows, with CUDA events:

- per call of the multi-leaf search, TorchSearch.leaf_actions + expand_backup_compact against expand_backup, on mid-game roots (a
  random-policy rollout first), after one warm-up search; a search is one single-leaf call and then 64 / L calls of L leaves, and only
  the L-leaf calls are timed.  The "network" is a fixed random scores tensor and zero values, so only library time is timed.  Dense
  configurations whose scores pass --max-dense-gb are skipped and say so.  The device bytes of both score tensors are recorded.
- TorchEnv.step_compact against step (GREEDY, f32) over --step-plies plies at --step-envs envs.
- TorchExamples.sample(compact=True) against sample() at --sample-batch rows (bf16 planes) from a ring filled by short searches.
- one whole move (TorchSearch.run, 65 simulations at 8 leaves) with two small networks on bf16 planes: a dense Linear(..., 8100) head, and
  an embedding-gather head that scores only the listed actions (compact=True).

Working sets: the dense score tensors of n >= 4,096 at L >= 8 (>= 1 GB) and the step's 65,536 x 8,100 f32 rows (2.1 GB) are larger than
the 126 MB L2; the compact rows at n = 4,096 (2 MB at L = 1) are not, and are read from L2 after the first call -- as they would be in
a self-play loop that hands the network's output straight to the library.  Prints one JSON object and writes it to --out with the GPU
name and power limit.

    python scripts/compact_bench.py --out profiles/compact_bench.json
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import cn_chess_ai_b200 as xq  # noqa: E402
from policy_ply_bench import gpu_info  # noqa: E402

SLOTS = 64


def _ev():
    return torch.cuda.Event(enable_timing=True)


def search_calls(n, L, reps, max_dense_gb, seed=7):
    dev = torch.device("cuda", 0)
    rows = n * L
    dense_gb = rows * 8100 * 4 / 1e9
    out = {"n": n, "leaves": L, "rows": rows, "dense_scores_bytes": rows * 8100 * 4, "compact_scores_bytes": rows * 128 * 4,
           "compact_actions_bytes": rows * 128 * 4 + rows}
    te = xq.TorchEnv(n, seed=seed)
    te.env.rollout_random(24)
    ts = xq.TorchSearch(te, 1 + SLOTS, L)
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    values = torch.zeros(rows, device=dev)
    calls = SLOTS // L
    for mode in ("compact", "dense"):
        if mode == "dense" and dense_gb > max_dense_gb:
            out["dense"] = f"skipped: scores tensor of {rows} rows x 8100 f32 ({dense_gb:.0f} GB) over --max-dense-gb {max_dense_gb}"
            continue
        scores = torch.randn((rows, 128 if mode == "compact" else 8100), generator=g, device=dev)
        tot = 0.0
        for rep in range(reps + 1):
            ts.reset()
            ts.select(1.5, 0.0)
            if mode == "compact":
                ts.leaf_actions()
                ts.expand_backup_compact(scores[:n], values[:n])
            else:
                ts.expand_backup(scores[:n], values[:n], view="side")
            ev = [(_ev(), _ev()) for _ in range(calls)]
            for c in range(calls):
                ts.select_leaves(L, 1.5, 0.0, 1.0) if L > 1 else ts.select(1.5, 0.0)
                ev[c][0].record()
                if mode == "compact":
                    ts.leaf_actions()
                    ts.expand_backup_compact(scores, values)
                else:
                    ts.expand_backup(scores, values, view="side")
                ev[c][1].record()
            torch.cuda.synchronize()
            if rep:
                tot += sum(a.elapsed_time(b) for a, b in ev) * 1e3
        out[f"{mode}_us_per_call"] = tot / (reps * calls)
        del scores
        torch.cuda.empty_cache()
    ts.close()
    te.close()
    torch.cuda.empty_cache()
    return out


def step(n, plies, reps, seed=3):
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    dense = torch.randn((n, 8100), generator=g, device=dev)
    comp = torch.randn((n, 128), generator=g, device=dev)
    out = {"envs": n, "plies": plies, "pick": "greedy", "dtype": "f32"}
    for mode in ("dense", "compact", "dense", "compact"):      # alternated: the second pair is the one recorded
        te = xq.TorchEnv(n, seed=seed)
        te.env.rollout_random(24)
        t = []
        for rep in range(reps + 1):
            a, b = _ev(), _ev()
            a.record()
            for _ in range(plies):
                if mode == "dense":
                    te.step(dense, pick="greedy")
                else:
                    te.step_compact(comp, pick="greedy")
            b.record()
            torch.cuda.synchronize()
            if rep:
                t.append(a.elapsed_time(b) * 1e3 / plies)
        out[f"{mode}_us_per_ply"] = sum(t) / len(t)
        te.close()
    a, b = _ev(), _ev()
    te = xq.TorchEnv(n, seed=seed)
    te.legal_actions()
    a.record()
    for _ in range(plies):
        te.legal_actions()
    b.record()
    torch.cuda.synchronize()
    out["legal_actions_us"] = a.elapsed_time(b) * 1e3 / plies
    te.close()
    return out


def sample(batch, reps, n=4096, seed=5):
    te = xq.TorchEnv(n, seed=seed)
    ts = xq.TorchSearch(te, 16)
    ex = xq.TorchExamples(ts, 1 << 16)
    dev = te.device

    def ev(planes):
        return torch.zeros((planes.shape[0], 8100), device=dev), torch.zeros(planes.shape[0], device=dev)
    for _ in range(4):
        ts.run(ev, 16)
        ex.record(ts)
        ts.play(1.0, 30)
    ex.end_games(torch.ones(n, dtype=torch.bool, device=dev), torch.zeros(n, device=dev))
    out = {"batch": batch, "ring_size": len(ex), "planes": "bf16"}
    for compact in (False, True, False, True):
        t = []
        for rep in range(reps + 1):
            a, b = _ev(), _ev()
            a.record()
            for i in range(20):
                ex.sample(batch, 1, i, compact=compact)
            b.record()
            torch.cuda.synchronize()
            if rep:
                t.append(a.elapsed_time(b) * 1e3 / 20)
        out[f"{'compact' if compact else 'dense'}_us_per_call"] = sum(t) / len(t)
    out["dense_policy_bytes"] = batch * 8100 * 4
    out["compact_policy_actions_bytes"] = batch * (128 * 4 + 128 * 4 + 1)
    for o in (ex, ts, te):
        o.close()
    return out


class _Trunk(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.body = torch.nn.Sequential(torch.nn.Conv2d(14, 32, 3, padding=1), torch.nn.ReLU(), torch.nn.Flatten(), torch.nn.Linear(32 * 90, 256),
                                        torch.nn.ReLU())
        self.value = torch.nn.Linear(256, 1)


def whole_move(n, L, reps, seed=7):
    """TorchSearch.run(65 simulations, leaves L): a dense Linear(256, 8100) head, and an embedding-gather head scoring only the listed
    actions (score = <h, E[action]>; the same parameter count)"""
    torch.manual_seed(0)
    trunk = _Trunk().cuda().to(torch.bfloat16)
    dense_head = torch.nn.Linear(256, 8100).cuda().to(torch.bfloat16)
    emb = torch.nn.Embedding(8101, 256).cuda().to(torch.bfloat16)

    def dense_eval(planes):
        with torch.no_grad():
            h = trunk.body(planes)
            return dense_head(h).float().contiguous(), torch.tanh(trunk.value(h).float()).reshape(-1)

    def compact_eval(planes, actions):
        with torch.no_grad():
            h = trunk.body(planes)
            e = emb(torch.where(actions >= 0, actions, 8100))            # [rows, 128, 256]
            return torch.bmm(e, h[:, :, None])[:, :, 0].float().contiguous(), torch.tanh(trunk.value(h).float()).reshape(-1)

    out = {"n": n, "leaves": L, "simulations": 1 + SLOTS, "network_calls": 1 + SLOTS // L}
    for mode in ("dense", "compact", "dense", "compact"):
        te = xq.TorchEnv(n, seed=seed)
        te.env.rollout_random(24)
        ts = xq.TorchSearch(te, 1 + SLOTS, L)
        times = []
        for rep in range(reps + 1):
            a, b = _ev(), _ev()
            a.record()
            if mode == "dense":
                ts.run(dense_eval, 1 + SLOTS, leaves=L)
            else:
                ts.run(compact_eval, 1 + SLOTS, leaves=L, compact=True)
            b.record()
            torch.cuda.synchronize()
            if rep:
                times.append(a.elapsed_time(b) * 1e3)
        out[f"{mode}_move_us"] = sum(times) / len(times)
        out[f"{mode}_move_us_min"] = min(times)
        ts.close()
        te.close()
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[4096, 65536])
    ap.add_argument("--leaves", type=int, nargs="+", default=[1, 8, 32])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--max-dense-gb", type=float, default=40.0)
    ap.add_argument("--step-envs", type=int, default=65536)
    ap.add_argument("--step-plies", type=int, default=20)
    ap.add_argument("--sample-batch", type=int, default=4096)
    ap.add_argument("--move-size", type=int, default=4096)
    ap.add_argument("--move-leaves", type=int, default=8)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    res = {"gpu": gpu_info(0), "reps": a.reps, "slots_per_search": SLOTS, "search": [], "step": None, "sample": None, "whole_move": None}
    for n in a.sizes:
        for L in a.leaves:
            r = search_calls(n, L, a.reps, a.max_dense_gb)
            res["search"].append(r)
            print(json.dumps(r), flush=True)
    res["step"] = step(a.step_envs, a.step_plies, a.reps)
    print(json.dumps(res["step"]), flush=True)
    res["sample"] = sample(a.sample_batch, a.reps)
    print(json.dumps(res["sample"]), flush=True)
    res["whole_move"] = whole_move(a.move_size, a.move_leaves, a.reps)
    print(json.dumps(res["whole_move"]), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
