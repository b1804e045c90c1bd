"""Timed legs of the DQN half of the metric (imported by bench.py)."""
import numpy as np

FLOP_PER_TRANSITION = 9_262_080      # fwd Q(s) + fwd Q'(s') + dense bwd of the {1260,128,8100} MLP (SURVEY 8d)


def _td_traffic():
    """DRAM bytes of one TD update from the ncu capture in profiles/ (None if the file is absent)"""
    import json
    import os
    p = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles", "traffic.json")
    return json.load(open(p)).get("td_update_dram_bytes_per_update") if os.path.exists(p) else None


ISSUED_FLOP_PER_UPDATE = {   # FLOPs the two tcgen05 kernels actually issue per batch-4096 update (the rest of the dense figure is skipped
    # exactly: one-hot input, one-hot TD error): row-max GEMM [4096 x 128] x [128 x 8100 -> 37 x 224] with the bias as a 9th K-step;
    # gradient contraction 11 row tiles x M128 x N256 (hi | lo) x K4096
    "l1_gemm_kernel": 2 * 4096 * (128 + 16) * 37 * 224, "dw_gemm_kernel": 2 * 11 * 128 * 256 * 4096}


def _gather_rows(net, vec, world, dist, dev, fused):
    """all ranks' copies of a small uint8 vector: through the library's own peer-memory all-gather when connected, else torch"""
    import torch
    if world == 1:
        return vec[None]
    if fused:
        return net.dist_allgather(vec)
    t = torch.from_numpy(vec).to(dev)
    g = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(g, t)
    return torch.stack(g).cpu().numpy()


def bench_dqn(stream, peaks, world=1, local=0, dist=None, envs=65536, replay_cap=1 << 20, batch=4096, updates=64, warmup=5, calls=5,
              train_loop=True):
    """BASELINE configs 3+4 on this rank: eps-greedy self-play with batched Q-net inference fills a 1M-transition
    replay ring, then batch-4096 TD updates (per GPU) are timed with CUDA events on `stream`: `calls` calls of `updates`
    sequential updates each (median / min over the calls, max over the ranks).  With world > 1 every update exchanges the
    compact gradient (inside the contraction kernel over peer memory, or NCCL with XQ_DIST=nccl) before the identical SGD
    step, and the run FAILS if the replicas' parameter bytes differ afterwards."""
    import torch
    from . import BatchedEnv, DQN, ReplayBuffer, collect, td_update_replay, td_update_replay_n
    import os
    from .dist import allreduce_sum_, connect_peers, grad_tensor
    dev = torch.device("cuda", local)
    rank = dist.get_rank() if dist is not None else 0
    env = BatchedEnv(envs, device=local, seed=31, env_id0=rank * envs)
    net = DQN((1260, 128, 8100), lr=1e-6, device=local, seed=31)
    rb = ReplayBuffer(replay_cap, device=local)
    env.set_stream(stream.cuda_stream)
    net.set_stream(stream.cuda_stream)
    plies = max(1, replay_cap // envs)
    collect(net, env, rb, 2, 0.1)                      # warm-up
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    collect(net, env, rb, plies, 0.1)
    b.record(stream)
    torch.cuda.synchronize()
    collect_ms = a.elapsed_time(b)
    fused = world > 1 and os.environ.get("XQ_DIST", "fused") != "nccl"
    if fused:
        connect_peers(net, dev)                        # from here on every applied update exchanges its gradient inside the contraction kernel
    grads = grad_tensor(net, dev) if world > 1 and not fused else None

    def one(i):
        if world > 1 and not fused:
            td_update_replay(net, rb, batch, 1000 + rank, i, True, 1e-6, apply=False)
            allreduce_sum_(grads)
            net.apply_grads(1e-6)
        else:
            td_update_replay(net, rb, batch, 1000 + rank, i, True, 1e-6, apply=True)

    for i in range(warmup):
        one(i)
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    pipelined = (world == 1 or fused) and os.environ.get("XQ_TD_PIPELINE", "1") != "0"
    if pipelined:
        td_update_replay_n(net, rb, batch, 1000 + rank, 10000, warmup, True, 1e-6)      # warm the second stream / both buffer slots
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(calls + 1)]
    evs[0].record(stream)
    for c in range(calls):
        if pipelined:  # one call = `updates` sequential updates (each with its gradient exchange when world > 1), the target-net branch of
            td_update_replay_n(net, rb, batch, 1000 + rank, warmup + c * updates, updates, True, 1e-6)      # update i+1 under the online branch of update i
        else:
            for i in range(updates):
                one(warmup + c * updates + i)
        evs[c + 1].record(stream)
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    per_call = [evs[c].elapsed_time(evs[c + 1]) for c in range(calls)]
    if fused and net.dist_timed_out():
        raise RuntimeError("gradient exchange: a peer never signalled (dist_timed_out)")
    # multi-GPU parity where the driver can see it: the replicas' parameter BYTES must be identical after the timed updates
    digests = _gather_rows(net, net.params_digest(), world, dist, dev, fused)
    replicas_identical = bool((digests == digests[0]).all())
    if not replicas_identical:
        raise RuntimeError("multi-GPU TD updates: the replicas' parameters differ after the timed updates (digest mismatch)")
    t = torch.tensor(per_call + [collect_ms], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    per_call, collect_ms = [float(x) for x in t[:calls]], float(t[calls])
    us = 1e3 * sum(per_call) / (updates * calls)
    us_sorted = sorted(1e3 * x / updates for x in per_call)
    tflops = FLOP_PER_TRANSITION * batch / (us * 1e-6) / 1e12          # per GPU
    issued = sum(ISSUED_FLOP_PER_UPDATE.values()) * (batch / 4096) / (us * 1e-6) / 1e12
    out = {"metric": "DQN TD updates/s (batch 4096 per GPU, target-net bootstrap, SGD applied)",
           "td_updates_per_s": 1e6 / us, "pipelined_over_two_streams": pipelined, "transitions_per_s": 1e6 / us * batch * world, "us_per_update": us,
           "us_per_update_median": us_sorted[len(us_sorted) // 2], "us_per_update_min": us_sorted[0], "us_per_update_calls": [1e3 * x / updates for x in per_call],
           "timed": "%d calls x %d sequential updates (%d kernel launches); mean over all, median / min over the calls, max over ranks" % (calls, updates, calls * updates * 4),
           "batch_per_gpu": batch, "replay_transitions_per_gpu": replay_cap,
           "grad_allreduce": ("inside the gradient contraction kernel over peer memory: reduce-scatter of the 16-row blocks to owner ranks + all-gather, flag-in-data lines"
                              if fused else "nccl all_reduce + apply kernel") if world > 1 else False,
           "replicas_identical": replicas_identical if world > 1 else None,
           "selfplay_eps_greedy_steps_per_s": envs * plies * world / (collect_ms * 1e-3), "selfplay_envs_per_gpu": envs,
           "roofline": {"bound": "tensor", "achieved": tflops, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s", "frac": tflops / peaks["bf16_tflops"],
                        "traffic": _td_traffic(), "peak_source": peaks["source"],
                        "issued": {"tflops": issued, "frac": issued / peaks["bf16_tflops"], "flop_per_update": ISSUED_FLOP_PER_UPDATE,
                                   "note": "FLOPs the two tcgen05 kernels issue (row-max GEMM incl. the bias K-step, gradient contraction hi|lo) / time of the whole update"},
                        "note": "achieved = ALGORITHMIC dense FLOPs (9,262,080 per transition) / time of the whole update (4 kernels chained by programmatic dependent launch, replay draws resolved in place); "
                                "the kernels exploit the one-hot input and one-hot TD error, so far fewer FLOPs are issued (DESIGN.md)"}}
    # self-play leg: per env per ply the acting path reads / writes the carried layer-0 sum (2 x 512 B), h(s) hi + lo (2 x 2 x 256 B), Q(s)[0..95]
    # (2 x 384 B), the env record (2 x 64 B), the remembered board (2 x 48 B) and writes the transition (128 B) = 3,168 B (DESIGN.md section 4)
    sp_bytes = 3168
    sp_gbs = envs * plies * sp_bytes / (collect_ms * 1e-3) / 1e9
    out["selfplay_roofline"] = {"bound": "hbm", "achieved": sp_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": sp_gbs / peaks["hbm_gbs"], "traffic": None,
                                "algorithmic_bytes_per_env_ply": sp_bytes, "us_per_ply": 1e3 * collect_ms / plies,
                                "note": "per GPU; the act kernel is bound by warp-instruction issue, the contraction by HBM (DESIGN.md section 4)"}
    if train_loop and (world == 1 or fused):
        # BASELINE config 4 end to end through the public episode driver (xq_train_run = the batched ChessAI::train), ONE call per rank:
        # rounds of [4 collector plies over all envs -> 64 batch-4096 TD updates, each exchanging its gradient at N > 1] (replay ratio 1),
        # the finished games of all ranks merged and drained to the host every round; wall clock around the whole call, host work included
        from .trainer import train
        import time
        train(net, env, rb, n_games=2000 * world, plies_per_round=4, updates_per_round=64, batch=batch, lr=1e-6, autosave_games=0)      # warm-up round
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        rep = train(net, env, rb, n_games=150000 * world, plies_per_round=4, updates_per_round=64, batch=batch, lr=1e-6, autosave_games=0)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt[0])
        d2 = _gather_rows(net, net.params_digest(), world, dist, dev, fused)
        if not bool((d2 == d2[0]).all()):
            raise RuntimeError("multi-GPU xq_train_run: the replicas' parameters differ after the run (digest mismatch)")
        out["train_loop"] = {"what": "xq_train_run, one call per rank: rounds of 4 eps-greedy plies x %d envs per GPU + 64 TD updates of batch %d per GPU (target-net bootstrap, "
                                     "target sync every 100 plies, gradient exchange per update at N > 1), games of all ranks merged per round; wall clock, max over ranks" % (envs, batch),
                             "seconds": dt, "rounds": rep["plies"] // 4, "ms_per_round": 1e3 * dt / max(1, rep["plies"] // 4), "games": rep["games"], "games_per_s": rep["games"] / dt,
                             "env_steps_per_s": rep["transitions"] / dt, "td_updates_per_s": rep["updates"] / dt, "trained_transitions_per_s": rep["updates"] * batch * world / dt,
                             "replicas_identical": True if world > 1 else None}
    env.close(); net.close(); rb.close()
    return out
