"""Times the Gumbel root search (xq_gumbel_*: TorchGumbel, TorchExamples.record_gumbel) against the PUCT calls of the same move, on
mid-game roots (a 24-ply random-policy rollout first) searched with 64 simulations of a fixed random f32 scores "network" and zero values,
as in search_bench.py, so that only library and torch time is timed.  CUDA events around every timed call:
  begin: TorchGumbel.begin on fresh roots (expansion of every root + the Gumbel draws), against the first PUCT select + expand_backup
    that expands the roots in a PUCT search;
  select: every select() call of a whole 64-simulation search, at 1 and 8 leaves per call, against TorchSearch.select / select_leaves
    of the same search shape (expand_backup between calls, not timed);
  root / play / record: TorchGumbel.root (dense pi' rows), TorchGumbel.play and TorchExamples.record_gumbel against TorchSearch.root,
    TorchSearch.play(temperature=1) and TorchExamples.record; the env's boards are restored between play calls (outside the events);
  move: one whole move of the self-play loop, advance -> run -> record -> play -> finish, Gumbel (TorchGumbel.run, record_gumbel) against
    PUCT with Dirichlet root noise (TorchSearch.run(dirichlet_alpha), record), at 1 and 8 leaves per call.
Prints one JSON object and writes it to --out, with the GPU name and power limit read in the same run.

    python scripts/gumbel_bench.py --sizes 4096 65536 --sims 64 --reps 10 --out profiles/gumbel_bench.json
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
from search_play_bench import boards_tensor, event_us  # noqa: E402

M, ALPHA, EPS, LEAVES = 16, 0.3, 0.25, 8


def timed(fn):
    """microseconds of one call of fn() between CUDA events"""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3


def stats(times):
    return {"mean": sum(times) / len(times), "min": min(times), "calls": len(times)}


def run(n, sims, reps, seed=7):
    dev = torch.device("cuda", 0)
    te = xq.TorchEnv(n, seed=seed)
    te.env.rollout_random(24)                    # mid-game roots
    ts = xq.TorchSearch(te, 2 * sims, LEAVES)
    tg = xq.TorchGumbel(ts, M)
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    pool = torch.randn((n * LEAVES, 8100), generator=g, device=dev)
    zeros = torch.zeros(n * LEAVES, device=dev)

    def evaluate(planes):
        return pool[:planes.shape[0]], zeros[:planes.shape[0]]

    boards = boards_tensor(te)
    saved = boards.clone()
    out = {"n": n, "sims": sims, "max_considered": M}

    # begin and the selections of whole searches
    t = {k: [] for k in ("gumbel_begin", "puct_first_select_expand", "gumbel_select_L1", "gumbel_select_L8", "puct_select_L1",
                         "puct_select_L8")}
    for r in range(reps + 1):
        for L in (1, LEAVES):
            ts.reset()
            tb = timed(lambda: tg.begin(pool[:n], zeros[:n], sims, seed=r))
            sel = []
            for k in [L] * (sims // L) + ([sims % L] if sims % L else []):
                sel.append(timed(lambda: tg.select(k)))
                ts.expand_backup(pool[:n * k], zeros[:n * k])
            ts.reset()

            def first():
                ts.select()
                ts.expand_backup(pool[:n], zeros[:n])
            tf = timed(first)
            psel = []
            i = 1
            while i < sims:
                k = min(L, sims - i)
                psel.append(timed(lambda: ts.select() if k == 1 else ts.select_leaves(k)))
                ts.expand_backup(pool[:n * k], zeros[:n * k])
                i += k
            if r:
                t[f"gumbel_select_L{L}"] += sel
                t[f"puct_select_L{L}"] += psel
                if L == 1:
                    t["gumbel_begin"].append(tb)
                    t["puct_first_select_expand"].append(tf)
    for k, v in t.items():
        out[k + "_us"] = stats(v)

    # root / play / record after a whole Gumbel search (the PUCT calls read the same trees)
    tg.run(evaluate, sims, seed=1, leaves=LEAVES)

    def restore():
        boards.copy_(saved)

    ex = xq.TorchExamples(ts, 1 << 20, 4 * reps + 8)
    out["gumbel_root_us"] = event_us(lambda: tg.root(), reps)
    out["puct_root_us"] = event_us(lambda: ts.root(), reps)
    out["gumbel_play_us"] = event_us(lambda: tg.play(), reps, restore)
    out["puct_play_tau1_us"] = event_us(lambda: ts.play(temperature=1.0, sample_plies=1000), reps, restore)
    restore()
    out["record_gumbel_us"] = event_us(lambda: ex.record_gumbel(tg), reps)
    out["record_us"] = event_us(lambda: ex.record(ts), reps)
    ex.close()

    # whole moves of the self-play loop
    for L in (1, LEAVES):
        for kind in ("gumbel", "puct"):
            restore()
            ex = xq.TorchExamples(ts, 1 << 20, reps + 2)
            state = {"first": True}

            def move():
                if not state["first"]:
                    ts.advance(sims)
                if kind == "gumbel":
                    tg.run(evaluate, sims, leaves=L, reset=state["first"])
                    ex.record_gumbel(tg)
                    ex.finish(tg.play())
                else:
                    ts.run(evaluate, sims, reset=state["first"], dirichlet_alpha=ALPHA, dirichlet_eps=EPS, leaves=L)
                    ex.record(ts)
                    ex.finish(ts.play(temperature=1.0, sample_plies=30))
                state["first"] = False

            out[f"{kind}_whole_move_L{L}_us"] = event_us(move, reps)
            ex.close()
    tg.close()
    ts.close()
    te.close()
    torch.cuda.empty_cache()
    for L in (1, LEAVES):
        out[f"whole_move_gumbel_over_puct_L{L}"] = out[f"gumbel_whole_move_L{L}_us"]["mean"] / out[f"puct_whole_move_L{L}_us"]["mean"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[4096, 65536])
    ap.add_argument("--sims", type=int, default=64)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    res = {"gpu": gpu_info(0), "sims_per_move": a.sims, "max_simulations": 2 * a.sims, "max_considered": M, "leaves": [1, LEAVES],
           "timed_calls": a.reps, "puct_dirichlet": {"alpha": ALPHA, "eps": EPS}, "results": []}
    for n in a.sizes:
        r = run(n, a.sims, a.reps)
        res["results"].append(r)
        print(json.dumps(r), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
