#!/usr/bin/env python
"""Cost of keeping the terminal rows of reset envs (keep_final / macm_bind_final) on the bench batch (4096 envs x 64
agents, 16 batches rotated): single steps with auto-reset, and K=32 rollouts that cross one episode boundary
(time_limit 0.5 s: every env finishes on step 31 of each episode), each with the final arrays unbound and bound,
alternated three times.  Prints one JSON line per measurement and the card it ran on."""
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "gym-macm_b200"))
import torch  # noqa: E402
import gym_macm  # noqa: E402
from gym_macm import _lib  # noqa: E402

dev = torch.device("cuda", 0)
E, N, R, K = 4096, 64, 16, 32
sims = [gym_macm.BatchedFlock(E, n_agents=[N], reward_mode="linear", device=dev, seed=1234 + r, time_limit=0.5,
                              auto_reset=True, keep_final=True) for r in range(R)]
assert sims[0].engine.info.done_step == 31
g = torch.Generator(device=dev)
g.manual_seed(99)
acts = torch.zeros((61, E, N, 4), dtype=torch.uint8, device=dev)
acts[..., :3] = torch.randint(0, 3, (61, E, N, 3), generator=g, device=dev, dtype=torch.uint8)
for k in range(40 * R):
    sims[k % R].engine.step(acts[(k // R + 7 * (k % R)) % 61])


def bind(on):
    for s in sims:
        if on:
            f = _lib.MacmFinalOut(**{n: t.data_ptr() for n, t in s.engine.final.items()})
            _lib.check(_lib.lib().macm_bind_final(s.engine._h, C.byref(f)))
        else:
            _lib.check(_lib.lib().macm_bind_final(s.engine._h, None))


def timed(fn, n):
    for rep in range(2):   # the first pass warms up
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for k in range(n):
            fn(k)
        e1.record()
        torch.cuda.synchronize()
    return 1e3 * e0.elapsed_time(e1) / n


plain = [sims[0].engine.rollout_buffers(K) for _ in range(2)]
finals = [sims[0].engine.rollout_buffers(K, ("obs", "nn_idx", "rewards", "collided", "done", "final_obs",
                                             "final_nn_idx", "final_env_state")) for _ in range(2)]
cases = [
    ("step + auto-reset", False, lambda k: sims[k % R].engine.step(acts[k % 61]), 31 * R, 1),
    ("step + auto-reset", True, lambda k: sims[k % R].engine.step(acts[k % 61]), 31 * R, 1),
    ("rollout K=32, per-step outputs", False, lambda k: sims[k % R].engine.rollout(acts[:K], K, None, 0, plain[k & 1]), 4 * R, K),
    ("rollout K=32, per-step outputs", True, lambda k: sims[k % R].engine.rollout(acts[:K], K, None, 0, plain[k & 1]), 4 * R, K),
    ("rollout K=32, per-step outputs + final_*", True,
     lambda k: sims[k % R].engine.rollout(acts[:K], K, None, 0, finals[k & 1]), 4 * R, K),
]
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip()
print(json.dumps({"card": card}))
for rep in range(3):
    for name, bound, fn, n, steps in cases:
        bind(bound)
        us = timed(fn, n) / steps
        print(json.dumps({"case": name, "finals_bound": bound, "us_per_step": round(us, 3), "rep": rep}))
