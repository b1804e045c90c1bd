#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native Xiangqi env + DQN hot path.

Metric (BASELINE.json): env steps/s (movegen + step + terminal/reward, random policy) -- and DQN TD
updates/s as the `dqn` object -- at 1/2/4/8 B200, next to the reference CPU path on the host cores.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--envs E] [--plies P] [--dump-outputs DIR]
  torchrun ... bench.py --gpus N ...          (one rank per GPU, env shards, no data-path collective)
  python bench.py --impl reference ...        (the reference's own ChessBoard path on the host cores)

One "step" = one fused rollout launch: P plies (default 200 = one full-length game) over the E envs of
this GPU (default 4096 = BASELINE configs[1]).  Scaling is weak: E envs per GPU.
Timing: W warm-up steps, then exactly K steps, each bracketed by CUDA events on the launching stream
(the library is pointed at torch's current stream), L2 flushed between steps outside the timed
intervals; barrier + synchronize on both sides; max over ranks.
--dump-outputs DIR writes what the timed steps hand their caller (see dump_outputs) as .npy files, so that two
builds can be compared output for output: the seeds are fixed, so the same arguments give the same inputs.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ALGO_BYTES_PER_STEP = 136   # read 64 B record + write 64 B record + 8 B outputs (SURVEY 8d, DESIGN.md)
DUMP_MAX_ENVS = 65536       # 416 B of dumped arrays per env: at most 27 MB


def dump_outputs(out_dir, boards, stats):
    """The boards after the last timed step (the 90 square codes and every other field of the record; a fixed, seeded sample of
    DUMP_MAX_ENVS envs when there are more, their indices in env_index) and the statistics of the timed steps, as float arrays."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    idx = np.arange(len(boards))
    if len(idx) > DUMP_MAX_ENVS:
        idx = np.sort(np.random.default_rng(0).choice(len(idx), DUMP_MAX_ENVS, replace=False))
    b = boards[idx]
    s = np.arange(90)
    out = {"env_index": idx.astype(np.float64), "board_squares": ((b["sq"][:, s >> 3] >> (4 * (s & 7))) & 15).astype(np.float32)}
    out.update({"board_" + f: b[f].astype(np.float64) for f in boards.dtype.names if f != "sq"})
    out.update({"stats_" + f: np.array([stats[f]], np.float64) for f in stats.dtype.names})
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d.get("bf16_tflops_sustained"),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def cpu_reference_leg(n_threads, plies_per_thread, seed=1):
    """the reference's own ChessBoard/ChessAI path (oracle/_ref, compiled unmodified) on the host cores,
    or the plain-C port when that build is absent.  Returns (steps_per_s, kind, sample description)."""
    import ctypes as C
    from oracle import loader as O
    R = O.ref()
    tot = C.c_long()
    if R is not None:
        s = R.ref_bench_rollout_random(n_threads, plies_per_thread, seed, C.byref(tot))
        kind = "reference"
        what = (f"{n_threads} threads x {plies_per_thread} random-policy plies each through the reference's own ChessBoard/ChessAI "
                "classes compiled unmodified (getAllValidActions -> movePiece -> evaluateBoard -> checkGameOver, reset on terminal)")
    else:
        L = O.oracle()
        s = L.xqo_bench_rollout_random(n_threads, 64, max(1, plies_per_thread // 64), seed, C.byref(tot))
        kind = "port"
        what = f"{n_threads} threads x 64 envs x {max(1, plies_per_thread // 64)} plies through oracle/xq_oracle.c (plain-C port)"
    return tot.value / s, kind, what, tot.value, s


def cpu_legs(cores):
    """BASELINE.md section 4 on this box's host cores, through the reference's own classes (oracle/_ref): env-only on 1 core; config (i)
    random policy + one CPU forward per ply on 1 core and on all cores; config (iii) epsilon-greedy with the CPU forward on 1 core;
    config (iv) one TD step per ply (ChessAI::train) with the network on 1 core.  Bounded samples (a few seconds each); plies/s."""
    import ctypes as C
    from oracle import loader as O
    R = O.ref()
    if R is None:
        return {"unavailable": "oracle/_ref is not built"}
    out = {}
    tot = C.c_long()
    s = R.ref_bench_rollout_random(1, 400000, 1, C.byref(tot))
    out["env_only_1_core"] = {"steps_per_s": tot.value / s, "sample": "400000 random-policy plies, 1 thread"}
    R.ref_bench_policy.restype = C.c_double
    R.ref_bench_policy.argtypes = [C.c_int, C.c_int, C.c_double, C.c_uint64, C.POINTER(C.c_long), C.POINTER(C.c_long)]
    for name, mode, nt, what in (("config_i_forward_per_ply_1_core", 0, 1, "configs[0]: random policy + one FP64 {1260,128,8100} forward per ply on the CPU"),
                                 ("config_i_forward_per_ply_all_cores", 0, cores, "the same, one independent board + network per thread"),
                                 ("config_iii_eps_greedy_1_core", 1, 1, "DQN::selectAction(eps = 0.1): a CPU forward on 90 % of the plies")):
        p, g = C.c_long(), C.c_long()
        s = R.ref_bench_policy(mode, nt, 4.0, 7, C.byref(p), C.byref(g))
        out[name] = {"steps_per_s": p.value / s, "threads": nt, "plies": p.value, "games": g.value, "seconds": s, "what": what,
                     "seconds_for_1000_games": 1000 * 153.25 / (p.value / s) if p.value else None}
    try:
        r = subprocess.run([sys.executable, "-m", "oracle.ref_train_bench", "2", "--cpu"], cwd=ROOT, capture_output=True, text=True, timeout=120)
        out["config_iv_td_step_per_ply_1_core"] = json.loads(r.stdout.strip().splitlines()[-1])
    except Exception as ex:
        out["config_iv_td_step_per_ply_1_core"] = {"unavailable": f"{type(ex).__name__}: {ex}"[:200]}
    return out


def reference_train_leg(games=3, timeout=240):
    """the reference's OWN training loop (ChessAI::train: batch 1, its own CUDA kernels from src/dqn.cu compiled unmodified when a GPU
    is visible, else the CPU definition of its NeuralNetwork) for a bounded number of games, in a subprocess (oracle/ref_train_bench.py)"""
    try:
        r = subprocess.run([sys.executable, "-m", "oracle.ref_train_bench", str(games)], cwd=ROOT, capture_output=True, text=True, timeout=timeout)
        return json.loads(r.stdout.strip().splitlines()[-1])
    except Exception as ex:      # a reported baseline, never a reason to lose the bench line
        return {"unavailable": f"{type(ex).__name__}: {ex}"[:200]}


def adapter_train_leg(games=3, timeout=240):
    """the drop-in single-board path: the C++ adapter's ChessAI::train (cn_chess_ai_b200/adapter/xq_adapter.hpp) compiled here with g++ against
    libxq_b200.so and run for a bounded number of games -- the counterpart of reference_train"""
    import tempfile
    try:
        pkg = os.path.join(ROOT, "cn_chess_ai_b200")
        exe = os.path.join(tempfile.mkdtemp(), "train_bench")
        subprocess.run(["g++", "-std=c++17", "-O2", "-o", exe, os.path.join(pkg, "adapter", "examples", "train_bench.cpp"), "-L" + pkg, "-lxq_b200",
                        "-Wl,-rpath," + pkg], check=True, capture_output=True, timeout=120)
        r = subprocess.run([exe, str(games)], capture_output=True, text=True, timeout=timeout, cwd=os.path.dirname(exe))
        return json.loads(r.stdout.strip().splitlines()[-1])
    except Exception as ex:
        return {"unavailable": f"{type(ex).__name__}: {ex}"[:200]}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    plies = args.ref_plies
    vals = []
    for _ in range(args.warmup):
        cpu_reference_leg(cores, max(1000, plies // 20))
    t_tot, n_tot, kind, what = 0.0, 0, None, None
    for _ in range(args.steps):
        v, kind, what, n, s = cpu_reference_leg(cores, plies)
        vals.append(v); t_tot += s; n_tot += n
    value = n_tot / t_tot
    line = {"impl": "reference", "metric": "env steps/s (movegen+step, random policy)", "value": value, "unit": "steps/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_tot / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": {"workload": f"BASELINE configs[1]: {args.envs} envs random-policy rollouts from the opening, {args.plies} plies per step",
                       "note": "CPU arm: each step is a bounded sample of that workload, one independent board per host thread"},
            "cpu_baseline": {"value": value, "unit": "steps/s", "cores": cores, "kind": kind, "sample": what},
            "e2e": {"value": value, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    if not args.no_dqn:      # the DQN half of the metric through the reference's own loop
        line["dqn"] = {"metric": "transitions trained/s through the reference's ChessAI::train (selectAction + movePiece + 2-3 forwards + backpropagate per ply)",
                       "reference_train": reference_train_leg()}
    emit(line)
    return 0


_REAL_STDOUT = None


def emit(line):
    """the one JSON line of this run, on the process's real stdout"""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--envs", type=int, default=4096, help="envs per GPU (BASELINE configs[1]: 4096)")
    ap.add_argument("--plies", type=int, default=200, help="plies per fused launch (= one step)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--ref-plies", type=int, default=250000, help="plies per host thread per step of the reference arm")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-aux", action="store_true")
    ap.add_argument("--no-dqn", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the boards and statistics of the timed steps to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    # stdout carries exactly ONE JSON line: libraries that write to fd 1 on their own (NCCL prints "NCCL version ..." there) are sent to
    # stderr for the whole run, and the line goes to the saved descriptor at the end
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import cn_chess_ai_b200 as xq

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the hot path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")      # stdout carries exactly one JSON line
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    L = xq.lib()
    stream = torch.cuda.current_stream()
    E, P = args.envs, args.plies
    env = xq.BatchedEnv(E, device=local, seed=2024, env_id0=rank * E)
    env.set_stream(stream.cuda_stream)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # > 126 MB L2

    # ---- device-resident leg: `value` ----
    for _ in range(args.warmup):
        env.rollout_random_async(P)
    env.stats(reset=True)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = L.xq_launch_count()
    evs = []
    for _ in range(args.steps):
        flush.fill_(1)                      # L2 flush, outside the timed interval
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        env.rollout_random_async(P)
        b.record(stream)
        evs.append((a, b))
    barrier()
    launches = L.xq_launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    ms = sum(a.elapsed_time(b) for a, b in evs)
    st = env.stats(reset=True)
    assert int(st["steps"]) == E * P * args.steps, "stats mismatch: kernel did not apply every ply"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, env.get_boards(), st)
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    total_steps = E * P * args.steps * world
    value = total_steps / (ms_max * 1e-3)

    # ---- end-to-end leg through the host-buffer C ABI: xq_env_rollout_random_io = set_boards -> rollout -> get_boards + stats ----
    host_in = np.zeros(E, dtype=xq.ENV_DTYPE)
    host_in[:] = env.get_boards()
    pin_in = torch.from_numpy(host_in.view(np.uint8)).pin_memory()
    pin_out = torch.empty_like(pin_in).pin_memory()
    recs_in = pin_in.numpy().view(xq.ENV_DTYPE)
    recs_out = pin_out.numpy().view(xq.ENV_DTYPE)
    # the C-ABI call itself, host pointers resolved once (what a C++ caller does): pinned boards in, pinned boards + statistics out
    pin_stats = torch.zeros(64, dtype=torch.uint8).pin_memory()
    stats_out = pin_stats.numpy().view(xq.STATS_DTYPE)
    p_in, p_out, p_stats = recs_in.ctypes.data, recs_out.ctypes.data, stats_out.ctypes.data

    def e2e_call():
        rc = L.xq_env_rollout_random_io(env.handle, p_in, P, p_out, None, p_stats)
        if rc != 0:
            raise RuntimeError(L.xq_last_error().decode())
        return int(stats_out[0]["steps"])

    for _ in range(2):
        e2e_call()
    barrier()
    t0 = time.perf_counter()
    e2e_steps = 0
    for _ in range(args.steps):
        e2e_steps += e2e_call()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_serial = e2e_steps * world / float(t.item())
    # The same step double-buffered (the way a data generator drives it): a SECOND handle of E envs with its own pinned buffers on the SAME
    # stream; the host submits the step of one handle before it waits for the step of the other (xq_env_rollout_random_io_submit / _wait),
    # so launch latency and the host's wake-up hide under the other handle's kernel.  Every step still moves its own boards host -> device
    # and boards + statistics device -> host; kernels of one stream never overlap.
    env_b = xq.BatchedEnv(E, device=local, seed=2025, env_id0=(world + rank) * E)
    env_b.set_stream(stream.cuda_stream)
    pin_in_b = pin_in.clone().pin_memory()
    pin_out_b = torch.empty_like(pin_in_b).pin_memory()
    pin_stats_b = torch.zeros(64, dtype=torch.uint8).pin_memory()
    stats_b = pin_stats_b.numpy().view(xq.STATS_DTYPE)
    hs = [(env.handle, p_in, p_out, p_stats, stats_out),
          (env_b.handle, pin_in_b.numpy().ctypes.data, pin_out_b.numpy().ctypes.data, stats_b.ctypes.data, stats_b)]

    def submit(k):
        if L.xq_env_rollout_random_io_submit(hs[k][0], hs[k][1], P, hs[k][2], None, hs[k][3]) != 0:
            raise RuntimeError(L.xq_last_error().decode())

    def wait(k):
        if L.xq_env_rollout_random_io_wait(hs[k][0]) != 0:
            raise RuntimeError(L.xq_last_error().decode())
        return int(hs[k][4][0]["steps"])

    def e2e_pipelined(n_steps):
        done = 0
        submit(0)
        for i in range(1, n_steps):
            submit(i & 1)
            done += wait((i - 1) & 1)
        return done + wait((n_steps - 1) & 1)

    e2e_pipelined(4)
    barrier()
    t0 = time.perf_counter()
    e2e_steps = e2e_pipelined(args.steps)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    assert e2e_steps == E * P * args.steps, "e2e: a step did not apply every ply"
    t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = e2e_steps * world / float(t.item())
    del env_b

    pk = peaks()
    kernel_ms = ms_max / args.steps
    achieved = ALGO_BYTES_PER_STEP * E * P / (kernel_ms * 1e-3) / 1e9
    traffic, inst_per_step = None, None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    tj = {}
    if os.path.exists(tp):
        tj = json.load(open(tp))
        if (E, P) == (4096, 200):       # the capture is of this workload
            traffic = tj.get("rollout_kernel_dram_bytes_per_launch")
        inst_per_step = tj.get("rollout_kernel_warp_inst_per_step")

    line = {"metric": "env steps/s (movegen+step, random policy)", "value": value, "unit": "steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": kernel_ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": {"workload": f"BASELINE configs[1]: {E} envs/GPU random-policy rollouts from the opening (legal-move gen + step + "
                                   f"terminal/reward), {P} plies per fused launch (= one step), auto-reset",
                       "envs_per_gpu": E, "plies_per_step": P, "l2": "flushed between timed steps (256 MiB fill)",
                       "parallelism": f"env-sharded x{world}, no data-path collective"},
            "e2e": {"value": e2e_value, "unit": "steps/s", "h2d_bytes_per_step": int(recs_in.nbytes),
                    "d2h_bytes_per_step": int(recs_out.nbytes) + 64,
                    "mode": "double-buffered: two handles of the same workload alternate on one stream, step i + 1 is submitted before step i is "
                            "waited for (xq_env_rollout_random_io_submit / _wait); every step copies its boards in and its boards + statistics out; "
                            "kernels never overlap",
                    "serial_value": e2e_serial,
                    "serial_note": "one xq_env_rollout_random_io call after the other on one handle (launch latency and host wake-up exposed)"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": achieved / pk["hbm_gbs"],
                         "traffic": traffic, "kernel": "rollout_team_kernel<4> (up to 9,472 envs; rollout_lane_kernel above: aux.config5)", "peak_source": pk["source"],
                         "algorithmic_bytes_per_launch": ALGO_BYTES_PER_STEP * E * P,
                         "note": "integer/latency-bound by design: boards stay on chip for all plies of a launch (DESIGN.md)"},
            "clocks": clocks}
    if inst_per_step and clocks and clocks.get("sm_mhz"):
        # the bound that actually binds this kernel (SURVEY 8d): warp-instruction issue slots, 148 SMs x 4 schedulers x SM clock
        issue_peak = 148 * 4 * clocks["sm_mhz"] * 1e6
        issued = value / world * inst_per_step
        line["roofline"]["secondary"] = {"bound": "warp-instruction issue", "achieved": issued, "peak": issue_peak, "unit": "warp-inst/s",
                                         "frac": issued / issue_peak, "warp_inst_per_env_step": inst_per_step,
                                         "alu_pipe_pct_of_peak": tj.get("rollout_kernel_alu_pipe_pct"),
                                         "source": "instructions per step from the ncu capture in profiles/ (smsp__inst_executed.sum / steps); "
                                                   "peak = 148 SMs x 4 schedulers x the SM clock sampled during the run",
                                         "note": "4096 envs = 512 warps on 592 schedulers, 128 of 148 SMs: every warp sits alone on its scheduler and a launch lasts as long as "
                                                 "one warp's 200 plies (~2,000 cycles per ply for ~640 instructions: fixed-latency dependencies 0.95, barrier 0.47 stalled "
                                                 "warps per issued instruction) -- the kernel is latency-bound, neither roofline binds (DESIGN.md section 4)"}

    # ---- timing hygiene (SURVEY 8d): >= 100 further launches of the same step, median / min of the per-launch times, max over ranks ----
    reps = max(100, args.steps)
    evs = []
    for _ in range(reps):
        flush.fill_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream); env.rollout_random_async(P); b.record(stream)
        evs.append((a, b))
    barrier()
    per = sorted(a.elapsed_time(b) for a, b in evs)
    t = torch.tensor([per[len(per) // 2], per[0], per[-1]], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    line["timing"] = {"launches": reps, "ms_per_step_median": float(t[0]), "ms_per_step_min": float(t[1]), "ms_per_step_max": float(t[2]),
                      "value_at_median": E * P * world / (float(t[0]) * 1e-3), "note": "a second timed region of the same step, L2 flushed before each launch"}
    env.stats(reset=True)

    if not args.no_aux:
        aux = {}
        # the traced mode of the same workload (the mode the parity tests check): every ply's (action, list size, flags, reward) written to HBM
        from cn_chess_ai_b200._lib import check
        for _ in range(3):
            check(L.xq_env_rollout_random_traced_async(env.handle, P, None))
        barrier()
        evs = []
        for _ in range(20):
            flush.fill_(1)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream); check(L.xq_env_rollout_random_traced_async(env.handle, P, None)); b.record(stream)
            evs.append((a, b))
        barrier()
        t = torch.tensor([sum(a.elapsed_time(b) for a, b in evs)], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        aux["traced_steps_per_s"] = E * P * 20 * world / (float(t[0]) * 1e-3)
        # API mode (what a drop-in caller of getAllValidActions -> movePiece does, src/chessai.cpp:347-368, src/chessboard.cpp:38-64), device-resident:
        # per ply three launches -- ordered lists materialised in HBM, random-policy pick from the list, step (movePiece + reward + terminal)
        aux["api_mode"] = {}
        for n_api, p_api in ((E, 200), (65536, 50)):
            ae = xq.BatchedEnv(n_api, device=local, seed=2024, env_id0=rank * n_api)
            ae.set_stream(stream.cuda_stream)
            for _ in range(5):
                ae.api_ply_device()
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            for _ in range(p_api):
                ae.api_ply_device()
            b.record(stream)
            barrier()
            t = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device="cuda")
            if dist is not None:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            sps = n_api * p_api * world / (float(t[0]) * 1e-3)
            aux["api_mode"][str(n_api)] = {"envs_per_gpu": n_api, "plies": p_api, "launches": 3 * p_api, "steps_per_s": sps, "us_per_ply": 1e3 * float(t[0]) / p_api,
                                           "roofline": {"bound": "hbm", "achieved": 215 * sps / world / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s",
                                                        "frac": 215 * sps / world / 1e9 / pk["hbm_gbs"], "algorithmic_bytes_per_step": 215, "traffic": None}}
            ae.close()
        # BASELINE config 5: 1M envs in total (1M / N per GPU), random policy, 32 plies per launch
        per_gpu = (1 << 20) // world
        big = xq.BatchedEnv(per_gpu, device=local, seed=7, env_id0=rank * per_gpu)
        big.set_stream(stream.cuda_stream)
        big.rollout_random_async(8)
        barrier()
        evs = []
        for _ in range(5):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream); big.rollout_random_async(32); b.record(stream)
            evs.append((a, b))
        barrier()
        t = torch.tensor([sum(a.elapsed_time(b) for a, b in evs)], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        aux["config5_1M_envs_steps_per_s"] = (1 << 20) * 32 * 5 / (float(t[0]) * 1e-3)
        c5 = aux["config5_1M_envs_steps_per_s"]
        c5_gbs = ALGO_BYTES_PER_STEP * c5 / world / 1e9
        aux["config5"] = {"envs_total": 1 << 20, "envs_per_gpu": per_gpu, "plies_per_launch": 32, "launches": 5, "steps_per_s": c5,
                          "kernel": "rollout_lane_kernel (one thread per board: squares in registers, bitboards also in a per-thread shared-memory view, piece tables in shared memory)",
                          "roofline": {"bound": "hbm", "achieved": c5_gbs, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": c5_gbs / pk["hbm_gbs"],
                                       "traffic": tj.get("lane_kernel_dram_bytes_per_launch") if world == 1 and os.path.exists(tp) else None,
                                       "algorithmic_bytes_per_launch": ALGO_BYTES_PER_STEP * per_gpu * 32, "peak_source": pk["source"]}}
        if os.path.exists(tp) and tj.get("lane_kernel_warp_inst_per_step") and clocks and clocks.get("sm_mhz"):
            ipeak = 148 * 4 * clocks["sm_mhz"] * 1e6
            issued = c5 / world * tj["lane_kernel_warp_inst_per_step"]
            aux["config5"]["roofline"]["secondary"] = {"bound": "warp-instruction issue", "achieved": issued, "peak": ipeak, "unit": "warp-inst/s", "frac": issued / ipeak,
                                                       "warp_inst_per_env_step": tj["lane_kernel_warp_inst_per_step"], "alu_pipe_pct_of_peak": tj.get("lane_kernel_alu_pipe_pct"),
                                                       "issue_active_pct_ncu": tj.get("lane_kernel_issue_active_pct"),
                                                       "note": "the integer ALU pipe issues one warp-instruction every two cycles per scheduler; with ~53 % of the instructions on it "
                                                               "the ALU pipe (86 % busy) and the issue slots (80 % active) bind together (ncu: profiles/r2c_ncu_lane_rollout_list_summary.csv)"}
        big.close()
        line["aux"] = aux

    if not args.no_dqn:
        # the DQN half of the metric: every rank takes part (gradient all-reduce at N > 1), rank 0 reports
        d = xq.bench_dqn(stream, pk, world=world, local=local, dist=dist)
        line["dqn"] = d
        if rank == 0 and world == 1 and not args.no_cpu_baseline:
            d["reference_train"] = reference_train_leg()      # the reference's own batch-1 loop on this box, next to transitions_per_s
            d["adapter_train"] = adapter_train_leg()          # the same loop through the drop-in adapter classes (one board, FP64 kernels of this library)
        launches_total = L.xq_launch_count()
        line["gpu_launches_total"] = int(launches_total)

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        v, kind, what, _, _ = cpu_reference_leg(cores, 400000)
        line["cpu_baseline"] = {"value": v, "unit": "steps/s", "cores": cores, "kind": kind, "sample": what, "legs": cpu_legs(cores)}

    if rank == 0:
        emit(line)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
