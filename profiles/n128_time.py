#!/usr/bin/env python
"""us per step of 128-agent flock envs (four agents per lane): 2048 envs x 128 agents = the headline's 262,144 agents.
Arguments: N, E, and `tdm` for two-team deathmatch envs of N agents instead (random moves and attacks)."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "gym-macm_b200"))
import torch
import gym_macm

dev = torch.device("cuda", 0)
N = int(sys.argv[1]) if len(sys.argv) > 1 else 128
E = int(sys.argv[2]) if len(sys.argv) > 2 else 2048
TDM = len(sys.argv) > 3 and sys.argv[3] == "tdm"
R, K = 8, 400
g = torch.Generator(device=dev)
g.manual_seed(9)
if TDM:
    sims = [gym_macm.BatchedTDM(E, n_agents=[N // 2, N - N // 2], device=dev, seed=70 + r) for r in range(R)]
else:
    sims = [gym_macm.BatchedFlock(E, n_agents=[N], reward_mode="linear", device=dev, seed=70 + r,
                                  start_spread=20.0 * (N / 64.0) ** 0.5) for r in range(R)]
acts = torch.zeros((31, E, N, 4), dtype=torch.uint8, device=dev)
acts[..., :3] = torch.randint(0, 3, (31, E, N, 3), generator=g, device=dev, dtype=torch.uint8)
if TDM:
    acts[..., 3] = torch.randint(0, 2, (31, E, N), generator=g, device=dev, dtype=torch.uint8)
pool = gym_macm.BatchPool(sims)
main = torch.cuda.current_stream(dev)
for rep in range(2):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for st in pool.streams:
        st.wait_stream(main)
    for k in range(K):
        pool.step(acts[(k // R + 7 * (k % R)) % 31])
    for st in pool.streams:
        main.wait_stream(st)
    e1.record()
    torch.cuda.synchronize()
info = sims[0].engine.info
print("%s N=%d E=%d: %.2f us per step, %.3g agent-steps/s; %d threads x %d blocks, %d B smem; overflow %s" % (
    "tdm" if TDM else "flock", N, E, 1e3 * e0.elapsed_time(e1) / K, E * N * K / (e0.elapsed_time(e1) * 1e-3),
    info.threads_per_block, info.blocks, info.smem_bytes_per_block, sims[0].overflow_count()))
