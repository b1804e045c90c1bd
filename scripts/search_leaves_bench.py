"""Times the multi-leaf selection of the batched tree search (TorchSearch.select_leaves) against one leaf per tree: per call and per leaf,
select, observe of the leaves (bf16 planes) and expand + backup, with CUDA events around every call of R whole searches (after one
warm-up search) on mid-game roots (a random-policy rollout first).  A search is one single-leaf call (which expands the root) and then
64 / L calls of L leaves each; only the L-leaf calls are timed.  The "network" is a fixed random [n * L, 8100] f32 scores tensor and zero
values, so that only library time is timed; configurations whose scores tensor passes --max-rows rows are skipped and say so.  Also
the share of duplicate slots, and one whole move (TorchSearch.run, 65 simulations) with a small torch network at L = 1 and L = 8.
Prints one JSON object and writes it to --out, with the GPU name and power limit.

    python scripts/search_leaves_bench.py --sizes 1 64 4096 65536 --leaves 1 2 4 8 16 32 --reps 3 --out search_leaves_bench.json
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

SLOTS = 64          # selected slots per search after the first, single-leaf simulation


def run(n, L, reps, max_rows, seed=7):
    dev = torch.device("cuda", 0)
    if n * L > max_rows:
        return {"n": n, "leaves": L, "skipped": f"scores tensor of {n * L} rows x 8100 f32 ({n * L * 8100 * 4 / 1e9:.0f} GB) over --max-rows"}
    sims = 1 + SLOTS
    te = xq.TorchEnv(n, seed=seed)
    te.env.rollout_random(24)                    # mid-game roots
    ts = xq.TorchSearch(te, sims, L)
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    scores = torch.randn((n * L, 8100), generator=g, device=dev)
    values = torch.zeros(n * L, device=dev)
    one_sc, one_val = scores[:n], values[:n]
    phases = ("select", "observe_bf16", "expand_backup")
    tot = dict.fromkeys(phases, 0.0)
    calls = SLOTS // L
    dup = total = 0
    for rep in range(reps + 1):
        ts.reset()
        ts.select(1.5, 0.0)
        ts.expand_backup(one_sc, one_val, 1.0, view="side")
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(calls)]
        st = []
        for c in range(calls):
            e = ev[c]
            e[0].record()
            sel = ts.select_leaves(L, 1.5, 0.0, 1.0) if L > 1 else ts.select(1.5, 0.0)
            e[1].record()
            ts.observe(torch.bfloat16, "side")
            e[2].record()
            ts.expand_backup(scores, values, 1.0, view="side")
            e[3].record()
            st.append(sel.status)
        torch.cuda.synchronize()
        if rep == 0:
            continue                             # warm-up search
        for e in ev:
            for k, p in enumerate(phases):
                tot[p] += e[k].elapsed_time(e[k + 1]) * 1e3
        s = torch.cat([x.reshape(-1) for x in st])
        dup += int((s == 4).sum())
        total += s.numel()
    k = reps * calls
    out = {"n": n, "leaves": L, "calls_per_search": calls, "bytes_per_tree": xq.search_bytes_per_tree(sims, L)}
    for p in phases:
        out[f"{p}_us_per_call"] = tot[p] / k
        out[f"{p}_ns_per_leaf"] = tot[p] / k / (n * L) * 1e3
    call = sum(tot.values()) / k
    out["library_us_per_call"] = call
    out["library_ns_per_leaf"] = call / (n * L) * 1e3
    out["duplicate_share"] = dup / total
    ts.close()
    te.close()
    del scores, values
    torch.cuda.empty_cache()
    return out


def whole_move(n, L, reps, seed=7):
    """one move of self-play search: TorchSearch.run(65 simulations) with a small conv network on bf16 planes"""
    torch.manual_seed(0)
    net = torch.nn.Sequential(torch.nn.Conv2d(14, 32, 3, padding=1), torch.nn.ReLU(), torch.nn.Flatten(),
                              torch.nn.Linear(32 * 90, 8101)).cuda().to(torch.bfloat16)

    def evaluate(planes):
        with torch.no_grad():
            out = net(planes)
        return out[:, :8100].contiguous(), torch.tanh(out[:, 8100].float())

    te = xq.TorchEnv(n, seed=seed)
    te.env.rollout_random(24)
    ts = xq.TorchSearch(te, 1 + SLOTS, L)
    times = []
    for rep in range(reps + 1):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ts.run(evaluate, 1 + SLOTS, leaves=L, virtual_loss=1.0)
        e1.record()
        torch.cuda.synchronize()
        if rep:
            times.append(e0.elapsed_time(e1) * 1e3)
    ts.close()
    te.close()
    torch.cuda.empty_cache()
    return {"n": n, "leaves": L, "simulations": 1 + SLOTS, "network_calls": 1 + SLOTS // L, "move_us": sum(times) / len(times),
            "move_us_min": min(times), "move_us_max": max(times)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[1, 64, 4096, 65536])
    ap.add_argument("--leaves", type=int, nargs="+", default=[1, 2, 4, 8, 16, 32])
    ap.add_argument("--move-sizes", type=int, nargs="+", default=[64, 4096])
    ap.add_argument("--move-leaves", type=int, nargs="+", default=[1, 8])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--max-rows", type=int, default=1 << 20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    res = {"gpu": gpu_info(0), "reps": a.reps, "slots_per_search": SLOTS, "virtual_loss": 1.0, "results": [], "whole_move": []}
    for n in a.sizes:
        for L in a.leaves:
            r = run(n, L, a.reps, a.max_rows)
            res["results"].append(r)
            print(json.dumps(r), flush=True)
    for n in a.move_sizes:
        for L in a.move_leaves:
            r = whole_move(n, L, a.reps)
            res["whole_move"].append(r)
            print(json.dumps(r), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
