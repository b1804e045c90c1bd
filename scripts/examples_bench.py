"""The self-play example buffer (xq_examples_*, TorchExamples): time per call of record, end_games and sample, each set against the
bytes the algorithm has to move and the 7.7 TB/s HBM3e figure of the B200 data sheet.

Set-up per size n: a TorchSearch of --sims simulations on n envs from harvested-like positions (the opening plus a few random plies),
driven by a fixed seeded random [n, 8100] score tensor and random values, so that the roots have realistic edge counts.
  record: --iters calls on the same trees after --warmup calls (the staging area is emptied before the timed window and is large enough
    for all of them, so every call writes n examples).  Bytes: per tree both 64-byte records, the root's node words, 10 bytes per edge
    (act, N, W) and the 864-byte example.
  end_games: every env first holds --game-len staged examples; each timed call ends a disjoint share of the envs (--shares), so every
    call commits share x n x game-len examples.  Bytes: 864 read + 864 written per committed example, plus the scan's per-env words.
  sample: batch --batch, bf16 planes, with and without the packed mask, on a full ring.  Bytes: the policy row (32,400), the planes
    (2,520), the mask (1,016, when asked), value / q / index, the record gathered and read again (128), the example read whole (864).
Times are CUDA events around the window divided by the calls (launch gaps included).  Prints one JSON object and writes it to --out,
with the GPU name and power limit read in the same run.

    python scripts/examples_bench.py --sizes 4096 65536 --out profiles/examples_bench.json
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
from cn_chess_ai_b200._lib import DTYPE_BF16, VIEW_SIDE_TO_MOVE  # noqa: E402
from policy_ply_bench import gpu_info  # noqa: E402

HBM = 7.7e12


def window(fn, iters, warmup, before=None):
    """mean time per call in microseconds: CUDA events around `iters` calls after `warmup` calls; before() runs once, untimed"""
    for _ in range(warmup):
        fn(-1)
    if before:
        before()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return 1e3 * e0.elapsed_time(e1) / iters


def row(us, nbytes):
    return {"us": us, "bytes": nbytes, "achieved_TBps": nbytes / (us * 1e-6) / 1e12, "share_of_hbm_peak": nbytes / (us * 1e-6) / HBM}


def bench(n, a):
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev)
    g.manual_seed(a.seed)
    te = xq.TorchEnv(n, seed=a.seed)
    for _ in range(6):                                                   # a few random plies from the opening
        te.step(scores=torch.randn((n, 8100), generator=g, device=dev), pick="sample")
    ts = xq.TorchSearch(te, a.sims)
    scores = torch.randn((n, 8100), generator=g, device=dev)
    values = torch.rand(n, generator=g, device=dev) * 2 - 1
    ts.run(lambda planes: (scores, values), a.sims)
    torch.cuda.synchronize()
    out = {"n": n}

    # record
    maxg = max(a.game_len, a.iters + a.warmup)
    tx = xq.TorchExamples(ts, a.capacity, maxg)
    B = tx.examples
    us = window(lambda i: B.record_device(ts.search), a.iters, a.warmup, before=lambda: B.discard_device())
    tx.end_games(torch.ones(n, dtype=torch.bool, device=dev), torch.zeros(n, device=dev))
    ne = tx.get(0, min(n, a.capacity))["n_edges"].astype("int64")
    edges = int(ne.mean() * n)
    out["mean_root_edges"] = float(ne.mean())
    out["record"] = row(us, n * (64 + 64 + 2 + 864) + edges * 10)
    out["record"]["note"] = "the trees' root rows and the staging area of one call fit in the 126 MB L2 at 4,096 envs"

    # end_games
    B.discard_device()
    for _ in range(a.game_len):
        B.record_device(ts.search)
    torch.cuda.synchronize()
    res = torch.rand(n, generator=g, device=dev) * 2 - 1
    out["end_games"] = []
    for share in a.shares:
        k = max(1, int(round(share * n)))
        calls = min(a.iters, n // k)
        masks = torch.zeros((calls, n), dtype=torch.uint8, device=dev)
        for i in range(calls):
            masks[i, i * k:(i + 1) * k] = 1
        none = torch.zeros(n, dtype=torch.uint8, device=dev)
        us = window(lambda i: B.end_games_device((none if i < 0 else masks[i]).data_ptr(), res.data_ptr()), calls, 1)
        r = row(us, k * a.game_len * 2 * 864 + n * (1 + 4 + 8 + 4))
        r.update({"share_ending": share, "envs_ending": k, "examples_committed_per_call": k * a.game_len, "calls": calls})
        out["end_games"].append(r)
        B.discard_device()                                               # every env holds game-len examples again
        for _ in range(a.game_len):
            B.record_device(ts.search)
        torch.cuda.synchronize()

    # sample
    info = tx.info()
    bt = a.batch
    planes = torch.empty((bt, 14, 10, 9), dtype=torch.bfloat16, device=dev)
    policy = torch.empty((bt, 8100), dtype=torch.float32, device=dev)
    value, q = torch.empty(bt, device=dev), torch.empty(bt, device=dev)
    mask = torch.empty((bt, 254), dtype=torch.int32, device=dev)
    index = torch.empty(bt, dtype=torch.int64, device=dev)
    out["ring_size_when_sampled"] = info["size"]
    out["sample"] = []
    for want_mask in (False, True):
        mp = mask.data_ptr() if want_mask else None
        us = window(lambda i: B.sample_device(bt, 5, i + 1000, VIEW_SIDE_TO_MOVE, planes.data_ptr(), DTYPE_BF16, policy.data_ptr(),
                                              value.data_ptr(), q.data_ptr(), mp, index.data_ptr()), a.iters, a.warmup)
        r = row(us, bt * (32400 + 2520 + (1016 if want_mask else 0) + 16 + 128 + 864))
        r.update({"batch": bt, "planes": "bf16", "mask": want_mask})
        out["sample"].append(r)
    tx.close()
    ts.close()
    te.close()
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[4096, 65536])
    ap.add_argument("--sims", type=int, default=64)
    ap.add_argument("--game-len", type=int, default=200, help="staged examples per env before end_games")
    ap.add_argument("--shares", type=float, nargs="+", default=[0.005, 0.1], help="share of the envs one end_games call ends")
    ap.add_argument("--capacity", type=int, default=1 << 21)
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--seed", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    res = {"gpu": gpu_info(0), "hbm_bytes_per_s_datasheet": HBM, "sims": a.sims, "game_len": a.game_len, "capacity": a.capacity,
           "iters": a.iters, "results": []}
    for n in a.sizes:
        r = bench(n, a)
        r["bytes_allocated"] = xq.examples_bytes(n, a.capacity, max(a.game_len, a.iters + a.warmup))
        res["results"].append(r)
        print(json.dumps(r), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
