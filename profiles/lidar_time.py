"""Time of macm_lidar (every agent's fan of closest-hit ray casts) at the sizes a swarm policy uses: CUDA events over
many launches after warm-up.

    python profiles/lidar_time.py [--iters 200]

Cases, each beside one step of the same batch: every agent of a 4096 x 64 Flock batch at 32 and 128 rays of 10 m, both
freshly spawned and gathered (after 300 steps of the `flock` actor); every agent of a 2048 x 128 Flock batch and of a
1024 x 45 TDM batch at 32 rays.  "kernel" launches macm_lidar alone; "lidar()" is the whole Python call.  The write
bound is the outputs' bytes (B*N*R fractions of 4 bytes and ids of 4 bytes) over 6448.7 GB/s, the HBM peak of the
roofline in DESIGN.md §3.  Outputs rotate over enough buffers to exceed the 126 MB L2, so each launch's stores reach
HBM.

Each case also times two launches that split its time:
  - every env index -1, which the kernel defines as a row of misses: nothing is staged or culled, only the stores run;
  - L = 0.01 m, where nothing but the caster's own disc (and a disc holding the origin) survives the cull: staging,
    the cull of every body, the float64 ray directions and the stores run, and next to no exact tests.
The full launch minus the second is the candidates' scatter and their exact tests.
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


def step_time(env, acts, iters):
    """One step of the batch, with its state put back afterwards (the scans below see the state as it was)."""
    import torch
    state = {n: t.clone() for n, t in env.engine.t.items()}
    t = timed(lambda k: env.engine.step(acts[k % len(acts)]), iters)
    for n, x in env.engine.t.items():
        x.copy_(state[n])
    torch.cuda.synchronize()
    return t


def case(name, env, n_rays, L, t_step, iters):
    import math
    import torch
    E, N = env.engine.E, env.engine.N
    fdt = env.engine.t["obs"].dtype
    nbytes = E * N * n_rays * (4 + 4)
    nbuf = max(2, -(-200_000_000 // nbytes))
    outs = [(torch.empty((E, N, n_rays), dtype=fdt, device=env.device),
             torch.empty((E, N, n_rays), dtype=torch.int32, device=env.device)) for _ in range(nbuf)]
    bad = torch.full((E,), -1, dtype=torch.int32, device=env.device)
    fov = 2 * math.pi
    eng = env.engine
    t_kernel = timed(lambda k: eng.lidar(E, n_rays, L, fov, None, *outs[k % nbuf]), iters)
    t_call = timed(lambda k: env.lidar(n_rays, L, out=outs[k % nbuf]), iters)
    t_miss = timed(lambda k: eng.lidar(E, n_rays, L, fov, bad, *outs[k % nbuf]), iters)
    t_short = timed(lambda k: eng.lidar(E, n_rays, 0.01, fov, None, *outs[k % nbuf]), iters)
    bound = nbytes / (HBM_GBS * 1e3)   # us
    print("%-36s R %4d  L %5.2f m  %7.1f MB  kernel %8.2f us (%6.0f M rays/s, %4.0f %% of the write bound %.1f us)  "
          "lidar() %8.2f us  scan / step %.2f" % (name, n_rays, L, nbytes / 1e6, t_kernel, E * N * n_rays / t_kernel,
                                                  100 * bound / t_kernel, bound, t_call, t_kernel / t_step))
    print("%-36s same launch: every env index -1 (stores only) %.2f us; L = 0.01 m (no candidates: staging, cull, "
          "directions, stores) %.2f us" % ("", t_miss, t_short))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    args = ap.parse_args()
    import torch
    import gym_macm
    assert torch.cuda.is_available(), "lidar_time.py measures on a CUDA device"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True)
    print(smi.stdout.strip().splitlines()[-1] if smi.returncode == 0 else "nvidia-smi: %s" % smi.stderr.strip())
    dev, it = "cuda:0", args.iters

    for N, E in ((64, 4096), (128, 2048)):
        env = gym_macm.BatchedFlock(E, n_agents=[N], device=dev, seed=1)
        acts = [env.pack_actions(torch.randint(0, 3, (E, N, 3), device=dev)).clone() for _ in range(8)]
        t_step = step_time(env, acts, it)
        print("Flock %d x %d fresh: step %.2f us" % (E, N, t_step))
        for R in ((32, 128) if N == 64 else (32,)):
            case("Flock %d x %d fresh, every agent" % (E, N), env, R, 10.0, t_step, it)
        if N == 64:
            for k in range(300):
                env.step(env.bot_actions("flock", seed=k))
            torch.cuda.synchronize()
            t_step = step_time(env, acts, it)
            print("Flock %d x %d gathered (300 flock steps): step %.2f us" % (E, N, t_step))
            for R in (32, 128):
                case("Flock %d x %d gathered, every agent" % (E, N), env, R, 10.0, t_step, it)
        env.close()

    tdm = gym_macm.BatchedTDM(1024, n_agents=[15, 15, 15], device=dev, seed=2)
    tdm.rollout(None, n_steps=120, policy="combat", want=())
    tacts = [tdm.bot_actions("combat", seed=k).clone() for k in range(8)]
    t_step = step_time(tdm, tacts, it)
    print("TDM 1024 x 45: step %.2f us, %d of %d agents dead" % (t_step, int((~tdm.alive).sum()), 1024 * 45))
    case("TDM 1024 x 45, every agent", tdm, 32, 10.0, t_step, it)


if __name__ == "__main__":
    main()
