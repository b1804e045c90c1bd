"""eps-greedy self-play collector timing (65,536 envs): us per ply"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import cn_chess_ai_b200 as xq
s = torch.cuda.current_stream()
for n in (65536, 16384, 262144):
    env = xq.BatchedEnv(n, seed=31); net = xq.DQN(lr=1e-6, seed=31); rb = xq.ReplayBuffer(1 << 20)
    env.set_stream(s.cuda_stream); net.set_stream(s.cuda_stream)
    xq.collect(net, env, rb, 4, 0.1)
    torch.cuda.synchronize()
    best = 1e9
    for _ in range(3):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(s); xq.collect(net, env, rb, 32, 0.1); b.record(s)
        torch.cuda.synchronize()
        best = min(best, a.elapsed_time(b))
    print(f"envs={n}: {1e3*best/32:.1f} us per ply = {n*32/(best*1e-3):.3e} steps/s")
    env.close(); net.close(); rb.close()
