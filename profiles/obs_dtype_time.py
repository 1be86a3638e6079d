#!/usr/bin/env python
"""Time per step at obs_dtype float32 / bfloat16 / float16, the three alternated in one run (median and range of the
repeats):

  tdm4      TDM config 4 (16,384 envs x 3 teams x 15 agents), device time per step (CUDA events), two batches in
            rotation (each batch's obs alone is 531 MB in fp32: nothing stays in L2)
  flock1    Flock config 1 (4096 envs x 64 agents, linear reward) on one stream, device time per step, 16 batches in
            rotation (> 2x L2)
  e2e       obs + rewards + done through the host-buffer path as bench.py's e2e leg does it: macm_step_host_async on
            3 batches in rotation, pinned host actions in, one device->host copy of the output slab per step,
            host clock around the whole loop
  peer      PeerGather (obs + rewards + done of every rank stored into rank 0's buffers by the step kernel), when run
            under torchrun with several GPUs; otherwise "not measured"

    python profiles/obs_dtype_time.py [--repeats 3]
    torchrun --nproc_per_node 8 profiles/obs_dtype_time.py        (adds the peer leg)
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "gym-macm_b200"))
import torch  # noqa: E402

import gym_macm  # noqa: E402

DTYPES = ("float32", "bfloat16", "float16")


def card():
    try:
        q = "name,power.limit,clocks.sm,clocks.max.sm"
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(","), [x.strip() for x in out.split(",")]))
    except Exception as ex:   # the numbers below are then unlabelled: say so
        return {"error": repr(ex)}


def device_ms(issue, n, streams=()):
    """ms per call of issue(k), k = 0..n-1, between CUDA events on the current stream (side streams joined)."""
    cur = torch.cuda.current_stream()
    for s in streams:
        s.wait_stream(cur)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(n):
        issue(k)
    for s in streams:
        cur.wait_stream(s)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def summary(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "repeats": len(xs)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--settle", type=int, default=64, help="untimed steps per batch after the spawn")
    ap.add_argument("--legs", default="tdm4,flock1,e2e,peer")
    args = ap.parse_args()
    legs = args.legs.split(",")
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    g = torch.Generator(device=dev)
    g.manual_seed(7)
    res = {"card": card() if rank == 0 else None, "world": world}

    def actions(pool, E, N, attack):
        a = torch.randint(0, 3, (pool, E, N, 4), generator=g, device=dev, dtype=torch.uint8)
        a[..., 3] = torch.randint(0, 2, (pool, E, N), generator=g, device=dev, dtype=torch.uint8) if attack else 0
        return a

    def settle(sims, acts):
        R = len(sims)
        for k in range(args.settle * R):
            sims[k % R].engine.step(acts[(k // R + 7 * (k % R)) % acts.shape[0]])
        torch.cuda.synchronize()

    def alternate(name, run):
        """run(dtype) -> number, for every dtype in turn, args.repeats rounds"""
        vals = {d: [] for d in DTYPES}
        for _ in range(args.repeats):
            for d in DTYPES:
                vals[d].append(run(d))
        res[name] = {d: summary(v) for d, v in vals.items()}

    if "tdm4" in legs and world == 1:
        E, N = 16384, 45
        acts = actions(17, E, N, True)
        sims = {d: [gym_macm.BatchedTDM(E, n_agents=[15, 15, 15], device=dev, seed=41 + r, obs_dtype=d) for r in range(2)]
                for d in DTYPES}
        for d in DTYPES:
            settle(sims[d], acts)

        def tdm(d):
            s = sims[d]
            issue = lambda k: s[k % 2].engine.step(acts[(k // 2 + 7 * (k % 2)) % 17])
            device_ms(issue, 8)
            return 1e3 * device_ms(issue, 100)
        alternate("tdm4_us_per_step", tdm)
        res["tdm4_obs_bytes_per_step"] = {d: int(sims[d][0].engine.sizes.obs) for d in DTYPES}
        del sims, acts
        torch.cuda.empty_cache()

    if "flock1" in legs and world == 1:
        E, N, R = 4096, 64, 16
        acts = actions(61, E, N, False)
        sims = {d: [gym_macm.BatchedFlock(E, n_agents=[N], reward_mode="linear", device=dev, seed=1234 + r, obs_dtype=d)
                    for r in range(R)] for d in DTYPES}
        for d in DTYPES:
            settle(sims[d], acts)

        def flock(d):
            s = sims[d]
            issue = lambda k: s[k % R].engine.step(acts[(k // R + 7 * (k % R)) % 61])
            device_ms(issue, 2 * R)
            return 1e3 * device_ms(issue, 1000)
        alternate("flock1_us_per_step", flock)
        del sims
        torch.cuda.empty_cache()

    if "e2e" in legs and world == 1:
        E, N, DEPTH, STEPS = 4096, 64, 3, 240
        acts = actions(4, E, N, False)
        host = [acts[i].cpu().pin_memory() for i in range(4)]
        want = ("obs", "rewards", "done")
        sims = {d: [gym_macm.BatchedFlock(E, n_agents=[N], reward_mode="linear", device=dev, seed=1234 + r, obs_dtype=d)
                    for r in range(DEPTH)] for d in DTYPES}
        for d in DTYPES:
            settle(sims[d], acts)

        def e2e(d):
            pp = sims[d]
            for s_ in pp:
                for k in range(3):
                    s_.engine.step_host(host[k % 4], want=want)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for k in range(STEPS):
                cur = pp[k % DEPTH].engine
                if k >= DEPTH:
                    cur.host_sync()
                    float(cur.pinned()["rewards"][0, 0])     # the host reads a result
                cur.step_host(host[k % 4], want=want, wait=False)
            for s_ in pp:
                s_.engine.host_sync()
            return E * N * STEPS / (time.perf_counter() - t0)
        alternate("e2e_agent_steps_per_s", e2e)
        res["e2e_d2h_bytes_per_step"] = {
            d: int(sum(sims[d][0].engine.pinned()[n].numel() * sims[d][0].engine.pinned()[n].element_size() for n in want))
            for d in DTYPES}
        del sims

    if "peer" in legs:
        if world == 1:
            res["peer"] = "not measured: one process (run under torchrun with several GPUs)"
        else:
            import torch.distributed as dist
            from gym_macm.dist import PeerGather
            dist.init_process_group("nccl", device_id=dev)
            E, N = 4096, 64
            acts = actions(31, E, N, False)
            sims, peer = {}, {}
            for d in DTYPES:
                sims[d] = [gym_macm.BatchedFlock(E, n_agents=[N], reward_mode="linear", device=dev,
                                                 seed=51 + 100 * rank + r, env_index_base=rank * E, obs_dtype=d)
                           for r in range(2)]
                settle(sims[d], acts)
                peer[d] = PeerGather(sims[d][0], world * E, learner=0, names=("obs", "rewards", "done"))
            ms = {d: [] for d in DTYPES}
            for _ in range(args.repeats):
                for d in DTYPES:
                    s, pg = sims[d], peer[d]
                    issue = lambda k: s[k % 2].engine.rollout(acts[(k // 2 + 7 * (k % 2)) % 31], 1, None, 0, pg.mine[k & 1])
                    device_ms(issue, 8)
                    dist.barrier()
                    ms[d].append(1e3 * device_ms(issue, 200))
            for d in DTYPES:
                peer[d].close()
            res["peer_us_per_step"] = {d: summary(v) for d, v in ms.items()}
            res["peer_bytes_into_learner_per_step"] = {
                d: (world - 1) * E * N * (16 // (1 if d == "float32" else 2) + 4) + (world - 1) * E for d in DTYPES}
            dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
