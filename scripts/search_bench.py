"""Times the batched tree search (xq_search_*) per simulation: select, observe of the leaves (bf16 planes), expand + backup and the whole
simulation, with CUDA events around every call of R whole searches (after one warm-up search) on mid-game roots (a random-policy rollout
first).  The "network" is a fixed random [n, 8100] f32 scores tensor and zero values, so that only library time is timed.  Yardstick:
xq_env_policy_step_device GREEDY at the same env count (same generator and score staging as expand + backup).  Prints one JSON object
and writes it to --out, with the GPU name and power limit.

    python scripts/search_bench.py --sizes 4096 65536 --sims 64 200 --reps 3 --out search_bench.json
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
from policy_ply_bench import gpu_info, timed  # noqa: E402


def run(n, sims, reps, seed=7):
    dev = torch.device("cuda", 0)
    per_tree = xq.search_bytes_per_tree(sims)
    free, _ = torch.cuda.mem_get_info(dev)
    if per_tree * n > 0.8 * free:
        return {"n": n, "sims": sims, "bytes_per_tree": per_tree, "skipped": f"needs {per_tree * n / 1e9:.1f} GB, {free / 1e9:.1f} GB free"}
    te = xq.TorchEnv(n, seed=seed)
    te.env.rollout_random(24)                    # mid-game roots
    ts = xq.TorchSearch(te, sims)
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    scores = torch.randn((n, 8100), generator=g, device=dev)
    values = torch.zeros(n, device=dev)
    phases = ("select", "observe_bf16", "expand_backup")
    tot = dict.fromkeys(phases, 0.0)
    whole = 0.0
    for rep in range(reps + 1):
        ts.reset()
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(sims)]
        for s in range(sims):
            e = ev[s]
            e[0].record()
            ts.select(1.5, 0.0)
            e[1].record()
            ts.observe(torch.bfloat16, "side")
            e[2].record()
            ts.expand_backup(scores, values, 1.0, view="side")
            e[3].record()
        torch.cuda.synchronize()
        if rep == 0:
            continue                             # warm-up search
        for e in ev:
            for k, p in enumerate(phases):
                tot[p] += e[k].elapsed_time(e[k + 1]) * 1e3
            whole += e[0].elapsed_time(e[3]) * 1e3
    k = reps * sims
    out = {"n": n, "sims": sims, "bytes_per_tree": per_tree, "device_bytes": per_tree * n}
    out.update({f"{p}_us": tot[p] / k for p in phases})
    out["simulation_us"] = whole / k
    out["simulations_per_s_all_trees"] = n * 1e6 / out["simulation_us"]
    # yardstick: the fused GREEDY ply at the same env count (its own envs, auto-reset keeps them in play)
    ty = xq.TorchEnv(n, seed=seed)
    ty.env.rollout_random(24)
    out["policy_step_greedy_us"] = timed(lambda: ty.step(scores, pick="greedy", view="side"), 50, 5)
    # nodes actually made: a sample of trees
    nodes = [len(ts.search.get_tree(i)[0]) for i in range(0, n, max(1, n // 16))]
    out["nodes_per_tree_sampled"] = sum(nodes) / len(nodes)
    ts.close()
    te.close()
    ty.close()
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[4096, 65536])
    ap.add_argument("--sims", type=int, nargs="+", default=[64, 200])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    res = {"gpu": gpu_info(0), "reps": a.reps, "results": []}
    for n in a.sizes:
        for s in a.sims:
            r = run(n, s, a.reps)
            res["results"].append(r)
            print(json.dumps(r), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
