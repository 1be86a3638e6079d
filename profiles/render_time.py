"""Time of macm_render at the sizes a user runs: CUDA events over many launches after warm-up.

    python profiles/render_time.py [--iters 200]

Cases: every env of a 4096 x 64 Flock batch at 84 x 84 with fitted views (beside one step of the same batch), 16
frames at 480 x 640, and every env of a 1024 x 45 TDM batch at 84 x 84.  "kernel" launches macm_render alone on views
computed once; "render()" is the whole BatchedFlock.render call (views fitted by torch on the device, then the
kernel).  The write bound is B*H*W*3 bytes over 6448.7 GB/s, the HBM peak of the roofline in DESIGN.md §3.
Outputs rotate over enough frame buffers to exceed the 126 MB L2, so each launch's stores reach HBM.

The first case also times the same launch on two kinds of view the kernel defines: a half-width of 0 (black frames: no
primitive is staged or culled, the stores alone) and views 1 km away from every agent (every primitive staged and
culled, nothing drawn).  Against the full launch they split its time into stores, staging + culling, and drawing.
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


def case(name, env, size, envs, iters, breakdown=False):
    import torch
    from gym_macm import render
    H, W = size
    idx, B = render.env_index(env, envs)
    views = render.fit_views(env, idx, size)
    pal = torch.from_numpy(render.palette(env)).to(env.device)
    nbuf = max(2, -(-200_000_000 // (B * H * W * 3)))
    outs = [torch.empty((B, H, W, 3), dtype=torch.uint8, device=env.device) for _ in range(nbuf)]
    t_kernel = timed(lambda k: env.engine.render(B, H, W, idx, views, pal, outs[k % nbuf]), iters)
    t_call = timed(lambda k: env.render(size, envs=idx, out=outs[k % nbuf]), iters)
    if breakdown:
        black, away = views.clone(), views.clone()
        black[:, 2] = 0.0
        away[:, 0] += 1000.0
        t_black = timed(lambda k: env.engine.render(B, H, W, idx, black, pal, outs[k % nbuf]), iters)
        t_away = timed(lambda k: env.engine.render(B, H, W, idx, away, pal, outs[k % nbuf]), iters)
    nbytes = B * H * W * 3
    bound = nbytes / (HBM_GBS * 1e3)   # us
    print("%-34s B=%5d %4dx%-4d  %7.1f MB  kernel %8.2f us (%9.0f frames/s, %4.0f %% of the write bound %.1f us)"
          "   render() %8.2f us" % (name, B, H, W, nbytes / 1e6, t_kernel, B / t_kernel * 1e6, 100 * bound / t_kernel,
                                    bound, t_call))
    if breakdown:
        print("%-34s same launch: black frames (stores only) %.2f us, views 1 km away (staging + cull, nothing drawn) "
              "%.2f us, fitted %.2f us" % ("", t_black, t_away, t_kernel))
    return t_kernel


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    args = ap.parse_args()
    import torch
    import gym_macm
    assert torch.cuda.is_available(), "render_time.py measures on a CUDA device"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True)
    print(smi.stdout.strip().splitlines()[-1] if smi.returncode == 0 else "nvidia-smi: %s" % smi.stderr.strip())
    dev = "cuda:0"

    env = gym_macm.BatchedFlock(4096, n_agents=[64], device=dev, seed=1)
    acts = [env.pack_actions(torch.randint(0, 3, (4096, 64, 3), device=dev)).clone() for _ in range(8)]
    for k in range(60):   # a stepped state: agents spread, contacts
        env.step(acts[k % 8])
    t_step = timed(lambda k: env.engine.step(acts[k % 8]), args.iters)
    t_r = case("Flock 4096 x 64, every env", env, (84, 84), None, args.iters, breakdown=True)
    print("%-34s step %8.2f us; render every env / step = %.2f" % ("", t_step, t_r / t_step))
    case("Flock 4096 x 64, 16 frames", env, (480, 640), range(16), args.iters)
    env.close()

    tdm = gym_macm.BatchedTDM(1024, n_agents=[15, 15, 15], device=dev, seed=2)
    tdm.rollout(None, n_steps=120, policy="combat", want=())
    case("TDM 1024 x 45, every env", tdm, (84, 84), None, args.iters)


if __name__ == "__main__":
    main()
