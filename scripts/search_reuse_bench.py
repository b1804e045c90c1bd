"""Subtree reuse in self-play (xq_search_advance, TorchSearch.advance): games from the opening, one search per move, the root's most-visited
move played with TorchEnv.step(pick="given").  Each move after the first runs advance(min_free) and then min_free simulations
(run(reset=False)); the comparison loop runs reset() and the same number of simulations instead.  Reports the advance kernel's time
(CUDA events around every advance call of R timed games, after one warm-up game), the nodes kept and the root visits carried over (mean,
spread, share of trees that kept a subtree), the root's edge visits when the move is chosen, and the time per move of both loops.

The "network" is a fixed seeded random [n, 8100] f32 score tensor and zero values, as in search_bench.py, so that only library time is
timed.  A real network concentrates its visits differently, which changes how much of the tree the played move carries over.  Prints one
JSON object and writes it to --out, with the GPU name and power limit.

    python scripts/search_reuse_bench.py --sizes 4096 65536 --moves 16 --sims 64 --max-sims 128 --out profiles/search_reuse_bench.json
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


def stats(x):
    x = torch.cat(x).double() if isinstance(x, list) else x.double()
    q = torch.quantile(x, torch.tensor([0.1, 0.5, 0.9], dtype=torch.float64, device=x.device)).tolist()
    return {"mean": x.mean().item(), "std": x.std().item(), "p10": q[0], "p50": q[1], "p90": q[2], "min": x.min().item(), "max": x.max().item()}


def play(n, moves, sims, max_sims, reuse, reps, seed):
    """reps + 1 games of `moves` moves on n envs (the first game warms up); per move the event time of the whole move and, with reuse,
    of the advance call; the kept counts and carried root visits of every advance; the root's edge visits at every decision"""
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    scores = torch.randn((n, 8100), generator=g, device=dev)
    values = torch.zeros(n, device=dev)

    def evaluate(planes):
        return scores, values

    te = xq.TorchEnv(n, seed=seed)
    ts = xq.TorchSearch(te, max_sims)
    adv_ms, move_ms, kept, carried, decided = [], [], [], [], []
    for rep in range(reps + 1):
        te.env.reset()
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(moves)]
        rep_kept, rep_carried, rep_decided = [], [], []
        for mv in range(moves):
            e = ev[mv]
            e[0].record()
            if reuse and mv > 0:
                k = ts.advance(sims)
            else:
                ts.reset()
                k = None
            e[1].record()
            if k is not None:                                             # not part of the move's time
                rep_kept.append(k)
                rep_carried.append(ts.root("side").visits.sum(1))      # the kept root's edge visits: N_node - 1 of the kept root
            e[2].record()
            root = ts.run(evaluate, sims, c_puct=1.5, view="side", reset=False)
            rep_decided.append(root.visits.sum(1))
            te.step(actions=root.best, pick="given", view="side")
            e[3].record()
        torch.cuda.synchronize()
        if rep == 0:
            continue                                                      # warm-up game
        for mv, e in enumerate(ev):
            move_ms.append(e[0].elapsed_time(e[1]) + e[2].elapsed_time(e[3]))
            if reuse and mv > 0:
                adv_ms.append(e[0].elapsed_time(e[1]))
        kept += rep_kept
        carried += rep_carried
        decided += rep_decided
    ts.close()
    te.close()
    torch.cuda.empty_cache()
    out = {"move_ms_mean": sum(move_ms) / len(move_ms), "root_edge_visits_at_decision": stats(decided)}
    if reuse:
        out["advance_calls_timed"] = len(adv_ms)
        out["advance_us"] = {"mean": 1e3 * sum(adv_ms) / len(adv_ms), "min": 1e3 * min(adv_ms), "max": 1e3 * max(adv_ms)}
        out["nodes_kept"] = stats(kept)
        out["trees_keeping_a_subtree"] = torch.cat(kept).gt(0).double().mean().item()
        out["root_visits_carried"] = stats(carried)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[4096, 65536])
    ap.add_argument("--moves", type=int, default=16)
    ap.add_argument("--sims", type=int, default=64, help="simulations per move, and advance's min_free")
    ap.add_argument("--max-sims", type=int, default=128)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--seed", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    res = {"gpu": gpu_info(0), "moves": a.moves, "sims_per_move": a.sims, "min_free": a.sims, "max_simulations": a.max_sims,
           "timed_games": a.reps, "results": []}
    for n in a.sizes:
        r = {"n": n, "bytes_per_tree": xq.search_bytes_per_tree(a.max_sims),
             "advance": play(n, a.moves, a.sims, a.max_sims, True, a.reps, a.seed),
             "reset": play(n, a.moves, a.sims, a.max_sims, False, a.reps, a.seed)}
        res["results"].append(r)
        print(json.dumps(r), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
