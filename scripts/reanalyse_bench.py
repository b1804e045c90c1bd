"""Reanalyse (TorchExamples.load / refresh / refresh_gumbel / reanalyse): time per call of the two library calls, each set against the
bytes it has to move and the 7.7 TB/s HBM3e figure of the B200 data sheet, and a whole reanalyse pass next to one self-play move.

Set-up per size m: m envs a few random plies from the opening and a search of --sims simulations on them, driven by the fixed
random-scores evaluator of search_play_bench.py / gumbel_bench.py (one seeded [m, 8100] score tensor and zero values, whatever the
planes), so that the comparison shows library time, not a network's.  A ring of --capacity examples is filled by recording those trees
until it has wrapped; the reanalysed slots are m distinct random slots.
  load: --iters calls after --warmup.  Bytes per row: the index (8), the slot's record read (64) and the env's record written (64).
  refresh / refresh_gumbel: --iters calls on the same trees and slots (every call rewrites them, as the claim words are restored).  Bytes
    per row: the index read by both kernels (16), the claim word (atomic, read and restored: 12), the root's and the slot's records
    (128), the root's expanded and n_edges bytes (2), 10 bytes per root edge (act, N, W), action / visits (768), n_edges / q /
    total_visits (9) and the status (1).  refresh_gumbel also runs the improved-policy weights kernel, as record_gumbel does: its
    time is in the call, its bytes are not counted.
  reanalyse: TorchExamples.reanalyse of m slots (load, TorchSearch.run of --sims simulations with a reset, refresh), next to one
    self-play move of m envs with the same evaluator and simulations (TorchSearch.run with a reset, record, play, finish).  The share of
    the pass spent in the two library calls is (load + refresh) / reanalyse.
Times are CUDA events around the window divided by the calls (launch gaps included).  Prints one JSON object and writes it to --out,
with the GPU name and power limit read in the same run.

    python scripts/reanalyse_bench.py --sizes 4096 65536 --out profiles/reanalyse_bench.json
"""
import argparse
import json
import math
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import cn_chess_ai_b200 as xq  # noqa: E402
from examples_bench import HBM, row, window  # noqa: E402
from policy_ply_bench import gpu_info  # noqa: E402


def bench(m, a):
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev)
    g.manual_seed(a.seed)
    scores = torch.randn((m, 8100), generator=g, device=dev)
    values = torch.zeros(m, device=dev)

    def evaluate(planes):
        return scores, values

    te = xq.TorchEnv(m, seed=a.seed)
    for _ in range(6):                                                   # a few random plies from the opening
        te.step(scores=torch.randn((m, 8100), generator=g, device=dev), pick="sample")
    ts = xq.TorchSearch(te, a.sims)
    ts.run(evaluate, a.sims)
    per = min(64, math.ceil((a.capacity + m) / m))                      # records per commit, commits until the ring has wrapped
    tx = xq.TorchExamples(te, a.capacity, per)
    ones, zeros = torch.ones(m, dtype=torch.bool, device=dev), torch.zeros(m, device=dev)
    for _ in range(math.ceil((a.capacity + m) / (m * per))):
        for _ in range(per):
            tx.record(ts)
        tx.end_games(ones, zeros)
    info = tx.info()
    assert info["total_committed"] > a.capacity and info["size"] == a.capacity
    ne = tx.get(0, min(m, a.capacity))["n_edges"].astype(np.int64)
    edges = int(ne.mean() * m)
    out = {"m": m, "mean_root_edges": float(ne.mean()), "ring_total_committed": info["total_committed"]}

    index = torch.from_numpy(np.random.default_rng(a.seed).choice(a.capacity, m, replace=False).astype(np.int64)).to(dev)
    te2 = xq.TorchEnv(m, seed=a.seed + 1)
    ts2 = xq.TorchSearch(te2, a.sims)
    tg = xq.TorchGumbel(ts2, a.considered)
    B = tx.examples
    status = torch.empty(m, dtype=torch.uint8, device=dev)

    out["load"] = row(window(lambda i: B.load_device(te2.env, index.data_ptr()), a.iters, a.warmup), m * (8 + 64 + 64))
    ts2.run(evaluate, a.sims)
    refresh_bytes = m * (16 + 12 + 128 + 2 + 768 + 9 + 1) + edges * 10
    out["refresh"] = row(window(lambda i: B.refresh_device(ts2.search, index.data_ptr(), status.data_ptr()), a.iters, a.warmup), refresh_bytes)
    out["refresh"]["all_refreshed"] = bool((status == 0).all())
    tg.run(evaluate, a.sims)
    out["refresh_gumbel"] = row(window(lambda i: B.refresh_gumbel_device(tg.gumbel, index.data_ptr(), status.data_ptr()), a.iters, a.warmup),
                                refresh_bytes)
    out["refresh_gumbel"]["all_refreshed"] = bool((status == 0).all())
    out["refresh_gumbel"]["note"] = "includes the improved-policy weights kernel; its bytes are not counted"

    out["reanalyse_us"] = window(lambda i: tx.reanalyse(ts2, evaluate, index, a.sims), a.passes, 2)
    sp = xq.TorchExamples(te, 4 * m, a.passes + 4)

    def move(i):
        ts.run(evaluate, a.sims)
        sp.record(ts)
        sp.finish(ts.play(temperature=1.0, sample_plies=30))

    out["self_play_move_us"] = window(move, a.passes, 2)
    out["library_share_of_reanalyse"] = (out["load"]["us"] + out["refresh"]["us"]) / out["reanalyse_us"]
    out["reanalyse_over_self_play_move"] = out["reanalyse_us"] / out["self_play_move_us"]
    for h in (sp, tx):
        h.close()
    tg.close()
    ts2.close()
    ts.close()
    te2.close()
    te.close()
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[4096, 65536])
    ap.add_argument("--sims", type=int, default=64)
    ap.add_argument("--considered", type=int, default=16, help="max_considered of the Gumbel search")
    ap.add_argument("--capacity", type=int, default=1 << 21)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--passes", type=int, default=20, help="timed reanalyse passes and self-play moves")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--seed", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    res = {"gpu": gpu_info(0), "hbm_bytes_per_s_datasheet": HBM, "sims": a.sims, "capacity": a.capacity, "iters": a.iters,
           "passes": a.passes, "results": []}
    for m in a.sizes:
        r = bench(m, a)
        res["results"].append(r)
        print(json.dumps(r), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
