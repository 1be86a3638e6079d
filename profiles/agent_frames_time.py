"""Time of macm_render_agents (every agent's own heading-up frame) at the sizes a pixel policy uses: CUDA events over
many launches after warm-up.

    python profiles/agent_frames_time.py [--iters 200] [--half-width 8]

Cases: every agent of a 4096 x 64 Flock batch at 16 x 16 and at 32 x 32 (beside one step of the same batch), and every
agent of a 1024 x 45 TDM batch at 32 x 32.  "kernel" launches macm_render_agents alone; "render_agents()" is the whole
Python call.  The write bound is B*N*H*W*3 bytes over 6448.7 GB/s, the HBM peak of the roofline in DESIGN.md §3.
Outputs rotate over enough frame buffers to exceed the 126 MB L2, so each launch's stores reach HBM.

Each case also times the same launch with every env index set to -1, which the kernel defines as N black frames per
row: nothing is staged, transformed or culled, only the tile loop and its stores run.  Against the full launch this
splits its time into stores and the rest (staging, per-frame transform and cull, drawing).
"""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "gym-macm_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

HBM_GBS = 6448.7


def timed(fn, iters, warmup=20):
    import torch
    for k in range(warmup):
        fn(k)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for k in range(iters):
        fn(k)
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1e3 / iters   # us per call


def case(name, env, size, hw, iters):
    import torch
    from gym_macm import render
    H, W = size
    E, N = env.engine.E, env.engine.N
    pal = torch.from_numpy(render.palette(env)).to(env.device)
    nbytes = E * N * H * W * 3
    nbuf = max(2, -(-200_000_000 // nbytes))
    outs = [torch.empty((E, N, H, W, 3), dtype=torch.uint8, device=env.device) for _ in range(nbuf)]
    bad = torch.full((E,), -1, dtype=torch.int32, device=env.device)
    t_kernel = timed(lambda k: env.engine.render_agents(E, H, W, hw, None, pal, outs[k % nbuf]), iters)
    t_call = timed(lambda k: env.render_agents(size, hw, out=outs[k % nbuf]), iters)
    t_black = timed(lambda k: env.engine.render_agents(E, H, W, hw, bad, pal, outs[k % nbuf]), iters)
    bound = nbytes / (HBM_GBS * 1e3)   # us
    print("%-30s %4dx%-4d half-width %.1f m  %7.1f MB  kernel %8.2f us (%10.0f frames/s, %4.0f %% of the write bound "
          "%.1f us)   render_agents() %8.2f us" % (name, H, W, hw, nbytes / 1e6, t_kernel, E * N / t_kernel * 1e6,
                                                   100 * bound / t_kernel, bound, t_call))
    print("%-30s same launch, every env index -1 (black frames: the tile loop and its stores only) %.2f us" %
          ("", t_black))
    return t_kernel


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--half-width", type=float, default=8.0)
    args = ap.parse_args()
    import torch
    import gym_macm
    assert torch.cuda.is_available(), "agent_frames_time.py measures on a CUDA device"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True)
    print(smi.stdout.strip().splitlines()[-1] if smi.returncode == 0 else "nvidia-smi: %s" % smi.stderr.strip())
    dev, hw = "cuda:0", args.half_width

    env = gym_macm.BatchedFlock(4096, n_agents=[64], device=dev, seed=1)
    for k in range(60):   # a stepped state: the flock actor gathers agents, the random one spreads them; contacts
        env.step(env.bot_actions("flock" if k % 2 else "random", seed=k))
    acts = [env.pack_actions(torch.randint(0, 3, (4096, 64, 3), device=dev)).clone() for _ in range(8)]
    state = {n: t.clone() for n, t in env.engine.t.items()}
    t_step = timed(lambda k: env.engine.step(acts[k % 8]), args.iters)
    for n, t in env.engine.t.items():   # frames of the stepped state above, not of the timed steps' random walk
        t.copy_(state[n])
    torch.cuda.synchronize()
    print("Flock 4096 x 64: step %.2f us, %d of %d envs hold agents in a contact" %
          (t_step, int(env.collided.any(1).sum()), 4096))
    for size in ((16, 16), (32, 32)):
        t = case("Flock 4096 x 64, every agent", env, size, hw, args.iters)
        print("%-30s every agent's frame / step = %.2f" % ("", t / t_step))
    env.close()
    del state

    tdm = gym_macm.BatchedTDM(1024, n_agents=[15, 15, 15], device=dev, seed=2)
    tdm.rollout(None, n_steps=120, policy="combat", want=())
    tacts = [tdm.bot_actions("combat", seed=k).clone() for k in range(8)]
    state = {n: t.clone() for n, t in tdm.engine.t.items()}
    t_step = timed(lambda k: tdm.engine.step(tacts[k % 8]), args.iters)
    for n, t in tdm.engine.t.items():
        t.copy_(state[n])
    torch.cuda.synchronize()
    print("TDM 1024 x 45: step %.2f us, %d of %d agents dead" % (t_step, int((~tdm.alive).sum()), 1024 * 45))
    t = case("TDM 1024 x 45, every agent", tdm, (32, 32), hw, args.iters)
    print("%-30s every agent's frame / step = %.2f" % ("", t / t_step))


if __name__ == "__main__":
    main()
