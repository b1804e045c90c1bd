"""Times playing self-play moves from the search and drawing root noise in the library (xq_search_play_device,
xq_search_root_noise_device) against the torch compositions they replace, on mid-game roots (a 24-ply random-policy rollout first) searched
with 64 simulations of a fixed random [n, 8100] f32 scores "network" and zero values, as in search_bench.py, so that only library and
torch time is timed.  CUDA events around every timed call, R calls each after one warm-up call:
  play: TorchSearch.play greedy and at temperature 1 against root() (the dense [n, 8100] visits) -> pow / multinomial ->
    TorchEnv.step(pick="given"); the env's boards are restored between calls (outside the events) so that every call plays a real move;
  noise: TorchSearch.root_noise against the dense masked Dirichlet tensor built in torch (legal_mask, _standard_gamma, normalisation) and
    passed to advance(), which mixes it into the kept roots; advance() without noise is reported beside it;
  move: one whole move of the self-play loop, advance -> run(dirichlet_alpha) -> TorchExamples.record -> play -> finish.
Prints one JSON object and writes it to --out, with the GPU name and power limit read in the same run.

    python scripts/search_play_bench.py --sizes 4096 65536 --sims 64 --reps 20 --out profiles/search_play_bench.json
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

ALPHA, EPS = 0.3, 0.25


def event_us(fn, reps, before=None):
    """mean and min microseconds of fn() over reps calls after one warm-up call; before() runs outside the events"""
    times = []
    for r in range(reps + 1):
        if before:
            before()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        if r:
            times.append(e0.elapsed_time(e1) * 1e3)
    return {"mean": sum(times) / len(times), "min": min(times)}


def boards_tensor(te):
    """the env's device records as a uint8 [n, 64] tensor aliasing the library's array"""
    ptr, n = te.env.device_boards_ptr(), te.n

    class _B:
        __cuda_array_interface__ = {"shape": (n, 64), "typestr": "|u1", "data": (ptr, False), "version": 3, "strides": None}

    return torch.as_tensor(_B(), device=te.device)


def run(n, sims, reps, seed=7):
    dev = torch.device("cuda", 0)
    te = xq.TorchEnv(n, seed=seed)
    te.env.rollout_random(24)                    # mid-game roots
    ts = xq.TorchSearch(te, 2 * sims)
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    scores = torch.randn((n, 8100), generator=g, device=dev)
    values = torch.zeros(n, device=dev)

    def evaluate(planes):
        return scores, values

    ts.run(evaluate, sims)
    boards = boards_tensor(te)
    saved = boards.clone()

    def restore():
        boards.copy_(saved)

    out = {"n": n, "sims": sims}

    def torch_play(tau):
        def f():
            visits = ts.root("side").visits.float()
            w = visits if tau == 1.0 else visits.pow(1.0 / tau)
            w[:, 0] += (w.sum(1) == 0).float()   # a root without a visited edge (no legal action) would stop multinomial
            te.step(actions=torch.multinomial(w, 1).squeeze(1), pick="given", view="side")
        return f

    out["play_greedy_us"] = event_us(lambda: ts.play(temperature=0.0), reps, restore)
    out["play_tau1_us"] = event_us(lambda: ts.play(temperature=1.0, sample_plies=1000), reps, restore)
    out["torch_root_multinomial_step_tau1_us"] = event_us(torch_play(1.0), reps, restore)
    out["torch_root_pow_multinomial_step_tau0.5_us"] = event_us(torch_play(0.5), reps, restore)
    restore()

    # noise: the kernel, and the dense tensor built in torch and mixed by advance (the roots match their envs: every tree is kept)
    out["root_noise_us"] = event_us(lambda: ts.root_noise(ALPHA, EPS, seed=1), reps)
    conc = torch.full((n, 8100), ALPHA, device=dev)

    def torch_noise():
        mask = te.legal_mask(view="side")
        gam = torch._standard_gamma(conc) * mask
        ts.advance(sims, root_noise=gam / gam.sum(1, keepdim=True).clamp_min(1e-30), noise_eps=EPS)

    out["torch_dirichlet_advance_us"] = event_us(torch_noise, reps)
    out["advance_without_noise_us"] = event_us(lambda: ts.advance(sims), reps)

    # one whole move of the loop
    ex = xq.TorchExamples(ts, 1 << 20, reps + 2)
    state = {"first": True}

    def move():
        if not state["first"]:
            ts.advance(sims)
        ts.run(evaluate, sims, reset=state["first"], dirichlet_alpha=ALPHA, dirichlet_eps=EPS)
        ex.record(ts)
        ex.finish(ts.play(temperature=1.0, sample_plies=30))
        state["first"] = False

    out["whole_move_us"] = event_us(move, reps)
    ex.close()
    ts.close()
    te.close()
    torch.cuda.empty_cache()
    for a, b, name in (("torch_root_multinomial_step_tau1_us", "play_tau1_us", "play_speedup_tau1"),
                       ("torch_dirichlet_advance_us", "root_noise_us", "noise_speedup_vs_dense_advance")):
        out[name] = out[a]["mean"] / out[b]["mean"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[4096, 65536])
    ap.add_argument("--sims", type=int, default=64)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    res = {"gpu": gpu_info(0), "sims_per_move": a.sims, "max_simulations": 2 * a.sims, "timed_calls": a.reps, "alpha": ALPHA, "eps": EPS,
           "results": []}
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
