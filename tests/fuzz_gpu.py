#!/usr/bin/env python
"""Randomised parity sweep on a GPU box (not collected by pytest): random agent counts, densities, modes and solver
settings, every step of the CUDA path held to the oracle with the bars of tests/_parity.py; every few cases the same
configuration also goes through macm_rollout and is held to single steps.

    python tests/fuzz_gpu.py [--seconds 180] [--seed 1]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "gym-macm_b200"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

from _parity import compare_step, make_pair, overflow_bits, run_parity  # noqa: E402
from test_gpu_tdm import run_tdm  # noqa: E402


def rollout_case(rng, N, E, kw):
    import torch
    import gym_macm
    K = int(rng.integers(5, 60))
    seed = int(rng.integers(0, 1 << 30))
    one, many = [gym_macm.BatchedFlock(E, n_agents=[N], device="cuda:0", seed=seed, **kw) for _ in range(2)]
    if kw.get("action_mode") == "continuous":
        acts = (torch.rand((K, E, N, 2), device="cuda:0") * 2.4 - 1.2).contiguous()
    else:
        acts = torch.zeros((K, E, N, 4), dtype=torch.uint8, device="cuda:0")
        acts[..., :3] = torch.randint(0, 3, (K, E, N, 3), device="cuda:0", dtype=torch.uint8)
    per = []
    for k in range(K):
        one.step(acts[k])
        per.append((one.state["obs"].clone(), one.state["rewards"].clone(), one.state["nn_idx"].clone()))
    out = many.rollout(acts)
    torch.cuda.synchronize()
    assert torch.equal(out["obs"], torch.stack([p[0] for p in per]))
    assert torch.equal(out["rewards"], torch.stack([p[1] for p in per]))
    assert torch.equal(out["nn_idx"], torch.stack([p[2] for p in per]))
    for n in ("posvel", "angsleep", "fat", "contact_count", "env_state"):
        assert torch.equal(one.state[n], many.state[n]), n
    one.close()
    many.close()
    return K


def capacity(rng, N):
    """max_touching of a case: the library default (0), the shared-memory stage's 240, or full capacity N(N-1)/2,
    which is more than 240 from 23 agents on and then runs the kernels of macm_kernels_huge.cu."""
    return int(rng.choice([0, 240, N * (N - 1) // 2]))


def capped_case(rng, N, E, steps, spread, kw):
    """Capacities below full: every step, the overflow bits against the oracle's counts and every unflagged env held to
    the oracle (_parity.overflow_bits, compare_step's env mask).  Returns the number of envs flagged at the end."""
    import torch
    pairs = N * (N - 1) // 2
    C = int(rng.integers(max(1, pairs // 8), pairs + 1))
    mt = int(rng.choice([0, 16 * int(rng.integers(1, 16))]))
    env, ref, r2 = make_pair(E, N, None, int(rng.integers(0, 1 << 30)), spread, max_contacts=C, max_touching=mt, **kw)
    coord, rmode = kw.get("coord", "polar"), kw.get("reward_mode", "binary")
    cont = kw.get("action_mode", "discrete") == "continuous"
    ever, bits = np.zeros(E, int), np.zeros(E, int)
    for k in range(steps):
        if cont:
            act = r2.uniform(-1.2, 1.2, (E, N, 2)).astype(np.float32).astype(np.float64)
            env.step(torch.as_tensor(act, dtype=torch.float32, device="cuda:0"))
        else:
            act = r2.integers(0, 3, (E, N, 3))
            env.step(torch.as_tensor(act, device="cuda:0"))
        o = ref.flock_step(act)
        bits = overflow_bits(env, ref, bits, ever, k)
        compare_step(env, ref, o, k, coord, rmode, envs=bits == 0)
    env.close()
    return int((bits != 0).sum()), dict(max_contacts=C, max_touching=mt)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=180.0)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--tdm", type=float, default=0.2, help="share of team-deathmatch cases")
    args = ap.parse_args()
    rng = np.random.default_rng(args.seed)
    t0, cases, agent_steps, worst_tc, skipped = time.time(), 0, 0, 0, 0
    tdm_cases, deaths, capped, flagged = 0, 0, 0, 0
    # per build: the default kernels, or those of macm_kernels_huge.cu (max_touching above 240)
    by_build = {"default": {"flock": 0, "tdm": 0}, "huge": {"flock": 0, "tdm": 0}}
    while time.time() - t0 < args.seconds:
        if rng.random() < args.tdm:
            n_teams = int(rng.integers(2, 5))
            teams = [int(rng.integers(1, (128 if rng.random() < 0.2 else 64) // n_teams + 1)) for _ in range(n_teams)]
            side = float(rng.choice([3.0, 6.0, 12.0, 30.0]))
            N = sum(teams)
            mt = capacity(rng, N)
            desc = dict(kind="tdm", teams=teams, side=side, max_touching=mt)
            try:
                steps = int(rng.integers(100, 500))
                E = int(rng.choice([4, 24]))
                deaths += run_tdm(E, teams, steps, seed=int(rng.integers(0, 1 << 30)), width=side, height=side,
                                  attack_p=float(rng.choice([0.2, 0.5, 0.9])), check_every=int(rng.choice([1, 7])),
                                  max_touching=mt)
            except AssertionError as ex:
                if "overflow" in str(ex):
                    skipped += 1
                    continue
                print("MISMATCH", json.dumps(desc), str(ex)[:300], flush=True)
                sys.exit(1)
            tdm_cases += 1
            by_build["huge" if mt > 240 else "default"]["tdm"] += 1
            agent_steps += E * sum(teams) * steps
            continue
        N = int(rng.choice([2, 3, 4, 5, 6, 7, 8, 9, 12, 16, 17, 24, 31, 32, 33, 40, 45, 48, 63, 64, 65, 80, 100, 128]))
        E = int(rng.choice([3, 16, 40]))
        # side of the spawn square: from a pile (about one body area per agent) to the reference's 20 m
        spread = float(np.sqrt(N) * rng.choice([0.9, 1.3, 2.0, 3.5]) if rng.random() < 0.7 else 20.0)
        kw = dict(reward_mode=str(rng.choice(["binary", "linear"])), coord=str(rng.choice(["polar", "cartesian"])),
                  action_mode=str(rng.choice(["discrete", "discrete", "continuous"])),
                  damping_model=str(rng.choice(["taylor", "pade"])))
        if rng.random() < 0.3:
            kw.update(velocityIterations=int(rng.integers(1, 11)), positionIterations=int(rng.integers(0, 5)))
        if rng.random() < 0.15:
            kw.update(enableWarmStarting=False)
        targets = None
        if N >= 3 and rng.random() < 0.3:
            T = int(rng.integers(2, min(N, 5) + 1))
            targets = [int(i % T) for i in range(N)]
        steps = int(rng.integers(30, 160))
        policy = "random"
        if kw["action_mode"] == "discrete" and kw["coord"] == "polar" and rng.random() < 0.25:
            policy = str(rng.choice(["flock", "idle"]))
        if rng.random() < 0.25:   # capacities below full: the overflow flags and the isolation of the other envs
            desc = dict(N=N, E=E, spread=round(spread, 2), steps=steps, capped=True, **kw)
            try:
                f, caps = capped_case(rng, N, E, steps, spread, kw)
            except AssertionError as ex:
                print("MISMATCH", json.dumps(desc), str(ex)[:300], flush=True)
                sys.exit(1)
            capped += 1
            flagged += f
            agent_steps += E * N * steps
            continue
        mt = capacity(rng, N)
        desc = dict(N=N, E=E, spread=round(spread, 2), steps=steps, policy=policy, targets=targets, max_touching=mt, **kw)
        try:
            st = run_parity(E, N, steps, targets=targets, seed=int(rng.integers(0, 1 << 30)), spread=spread, policy=policy,
                            max_contacts=N * (N - 1) // 2, max_touching=mt, **kw)
            if cases % 4 == 0:
                rollout_case(rng, N, E, dict(kw, max_contacts=N * (N - 1) // 2, max_touching=mt))
        except AssertionError as ex:
            if "capacity overflow" in str(ex):
                # more than 240 touching contacts at once (an unphysical spawn pile: bodies that do not overlap cannot
                # exceed ~3N): outside the staged solver's range.  The device REPORTED it (the sticky flags
                # compare_step asserts on, BatchedFlock.overflowed / overflow_count); the case counts as reported,
                # its steps before the overflow were compared.
                skipped += 1
                continue
            print("MISMATCH", json.dumps(desc), str(ex)[:300], flush=True)
            sys.exit(1)
        cases += 1
        by_build["huge" if mt > 240 else "default"]["flock"] += 1
        agent_steps += E * N * steps
        worst_tc = max(worst_tc, st["max_touching"])
    print(json.dumps({"cases": cases, "tdm_cases": tdm_cases, "tdm_deaths_at_case_end": deaths, "agent_steps_checked": agent_steps, "max_touching_seen": worst_tc, "overflow_reported_by_device": skipped,
                      "capped_cases": capped, "capped_envs_flagged": flagged,
                      "cases_by_build": by_build,
                      "seconds": round(time.time() - t0, 1), "seed": args.seed}))


if __name__ == "__main__":
    main()
