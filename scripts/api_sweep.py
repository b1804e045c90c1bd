"""API-mode path on the device (lists -> pick -> step, three launches per ply): steps/s and per-kernel time; XQ_LEGAL_TEAM=0|1 forces the list kernel"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import cn_chess_ai_b200 as xq
from cn_chess_ai_b200._lib import check
s = torch.cuda.current_stream()
L = xq.lib()
sizes = ((4096, 200), (65536, 50), (1 << 20, 10))
if os.environ.get("XQ_SWEEP_SIZES"):      # e.g. "4096:200,8192:200"
    sizes = tuple(tuple(int(x) for x in t.split(":")) for t in os.environ["XQ_SWEEP_SIZES"].split(","))
for n, plies in sizes:
    env = xq.BatchedEnv(n, seed=7)
    env.set_stream(s.cuda_stream)
    for _ in range(20):
        env.api_ply_device()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(s)
    for _ in range(plies):
        env.api_ply_device()
    b.record(s)
    torch.cuda.synchronize()
    ms = a.elapsed_time(b)
    # the list kernel alone
    a.record(s)
    for _ in range(plies):
        env.legal_moves_device()
    b.record(s)
    torch.cuda.synchronize()
    ms_l = a.elapsed_time(b)
    a.record(s)
    for _ in range(plies):
        check(L.xq_env_step_device(env.handle, None, 1, None, None, None, None, None))
    b.record(s)
    torch.cuda.synchronize()
    ms_s = a.elapsed_time(b)
    print(f"team={os.environ.get('XQ_LEGAL_TEAM','auto')} envs={n}: api ply {1e3*ms/plies:.1f} us = {n*plies/(ms*1e-3):.3e} steps/s; list kernel {1e3*ms_l/plies:.1f} us ({321*n/(ms_l/plies*1e-3)/1e9:.0f} GB/s of 64+257 B/env); step kernel {1e3*ms_s/plies:.1f} us")
    env.close()
