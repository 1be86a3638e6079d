"""bench.py --dump-outputs: the outputs of the last timed step, from seeded inputs, so that two builds can be
compared output for output.  --steps is the number of timed steps (one launch each)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = {"obs", "rewards", "done", "nn_idx", "collided", "env_index"}
E, N, ROT, SETTLE, WARMUP = 256, 64, 2, 4, 3


def _bench(steps, out):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", str(WARMUP),
           "--envs", str(E), "--rot", str(ROT), "--settle", str(SETTLE), "--no-legs", "--e2e-steps", "0",
           "--cpu-seconds", "0.2", "--dump-outputs", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    res = json.loads(r.stdout.strip().splitlines()[-1])
    assert set(os.listdir(out)) == {n + ".npy" for n in NAMES}
    return res, {n: np.load(os.path.join(out, n + ".npy")) for n in NAMES}


def _replay(steps):
    """bench.py's inputs stepped serially here: batch r seeded 1234 + r, the action pool of generator seed 99, step k
    on batch k % ROT with pool entry (k // ROT + 7 (k % ROT)) mod 61; settle, warm-up, then the timed steps."""
    import torch
    import gym_macm
    dev = torch.device("cuda", 0)
    sims = [gym_macm.BatchedFlock(E, n_agents=[N], reward_mode="linear", device=dev, seed=1234 + r) for r in range(ROT)]
    g = torch.Generator(device=dev)
    g.manual_seed(99)
    acts = torch.zeros((61, E, N, 4), dtype=torch.uint8, device=dev)
    acts[..., :3] = torch.randint(0, 3, (61, E, N, 3), generator=g, device=dev, dtype=torch.uint8)
    for n_steps in (SETTLE * ROT, WARMUP, steps):
        for k in range(n_steps):
            sims[k % ROT].engine.step(acts[(k // ROT + 7 * (k % ROT)) % 61])
    torch.cuda.synchronize()
    last = sims[(steps - 1) % ROT]
    out = {n: last.state[n].cpu().numpy() for n in last.engine.OUTPUTS}
    for s in sims:
        s.close()
    return out


def test_dump_is_repeatable_and_follows_steps(tmp_path):
    res, a = _bench(5, tmp_path / "a")
    assert res["steps"] == 5 and res["gpu_launches"] == 5
    for n, x in a.items():
        assert x.dtype in (np.float32, np.float64), n
    assert a["obs"].shape == (E, N, 4) and a["rewards"].shape == (E, N) and a["done"].shape == (E,)
    assert np.array_equal(a["env_index"], np.arange(E))
    _, b = _bench(5, tmp_path / "b")
    for n in NAMES:
        assert np.array_equal(a[n], b[n]), n
    # 5 timed steps end on batch 0, 6 on batch 1: each dump is that batch after exactly that many steps
    res, c = _bench(6, tmp_path / "c")
    assert res["steps"] == 6 and res["gpu_launches"] == 6
    for steps, got in ((5, a), (6, c)):
        want = _replay(steps)
        for n, w in want.items():
            assert np.array_equal(got[n], w.astype(got[n].dtype)), (steps, n)
