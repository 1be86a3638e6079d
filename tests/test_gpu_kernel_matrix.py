"""Every step kernel the library dispatches, held to the oracle.

A sim runs one of six (lanes per env G, agents per lane APL) shapes for each env kind (DISPATCH_SHAPE in
macm_kernels.cu), in one of two builds: the default one, and the one of macm_kernels_huge.cu that a sim gets when
max_touching exceeds the 240 contacts of the shared-memory solver stage.  One-env-per-warp shapes (G = 32) also
have a wide launch, one block per SM that stages the sin/cos table in shared memory; it is chosen for large batches
and forced here with MACM_BLOCK_THREADS.  Each case below names the kernel it is meant to reach, asserts from the
launch info that it did, and steps it against the oracle from spawns that mix a dense pile (more touching contacts
than lanes: the level-scheduled solver) with sparser worlds.  Twins of each case are stepped with multi-step
rollouts and with one-step rollouts that write per-step outputs; both must equal the single steps bit for bit.
"""
import os

import numpy as np
import pytest

from _parity import compare_obs, compare_step, oracle_kwargs
from test_gpu_rollout import _same_state
from test_gpu_tdm import compare_tdm_step, tdm_spawn

pytestmark = pytest.mark.gpu

SHAPES = ((4, 1), (8, 1), (16, 1), (32, 1), (32, 2), (32, 4))
RAGGED_N = {(4, 1): 3, (8, 1): 7, (16, 1): 13, (32, 1): 29, (32, 2): 50, (32, 4): 113}
# Wide blocks: the shape's launch bound (896 threads, 448 with four agents per lane), unless the 227 KB of shared
# memory cannot hold that many envs' stages plus the table.  In the huge build the shared stage holds 240 touching
# contacts, so 64- and 128-slot envs fit 21 and 13 to a block.
WIDE_THREADS = {("default", 1): 896, ("default", 2): 896, ("default", 4): 448,
                ("huge", 1): 896, ("huge", 2): 672, ("huge", 4): 416}
# default-build max_touching: 240 where blocks are narrow; for wide blocks the largest capacity that still fits
DEFAULT_WIDE_TOUCHING = {1: 240, 2: 144, 4: 192}

FLOCK_A = dict(reward_mode="binary", coord="polar", action_mode="discrete", damping_model="pade")
FLOCK_B = dict(reward_mode="linear", coord="cartesian", action_mode="continuous", damping_model="taylor",
               velocityIterations=5, positionIterations=2, enableWarmStarting=False)


def _teams(N):
    # uneven splits: two teams below 8 agents, three above
    if N < 8:
        return [N - N // 2, N // 2] if N > 2 else [1, 1]
    a = (N + 2) // 3 + 2
    b = (N - a) // 2 + 1
    return [a, b, N - a - b]


# side of the pile arena per (kind, build / launch, N), found with the oracle: more touching contacts than lanes, at
# most about 80 % of the default build's max_touching, and more than 240 in the huge build from 50 agents on
PILE = {
    ("flock", "narrow"): {3: 0.6, 4: 0.6, 7: 1.2, 8: 1.2, 13: 2.0, 16: 2.0, 29: 2.4, 32: 2.8, 50: 4.6, 64: 5.8,
                          113: 10.0, 128: 11.8},
    ("flock", "wide"): {29: 2.8, 50: 6.2, 113: 11.8},
    ("flock", "huge"): {29: 1.1, 50: 2.6, 113: 4.4},
    ("tdm", "narrow"): {3: 0.6, 4: 0.6, 7: 3.4, 8: 2.2, 13: 2.0, 16: 1.4, 29: 2.2, 32: 2.8, 50: 5.4, 64: 7.8,
                        113: 13.2, 128: 15.0},
    ("tdm", "wide"): {29: 2.4, 50: 7.2, 113: 15.2},
    ("tdm", "huge"): {29: 0.8, 50: 1.6, 113: 3.0},
}


def _cases():
    out = []
    for build, wide, shapes in (("default", False, SHAPES), ("default", True, SHAPES[3:]),
                                ("huge", False, SHAPES[3:]), ("huge", True, SHAPES[3:])):
        for G, APL in shapes:
            ns = [RAGGED_N[(G, APL)]]
            if build == "default" and not wide:
                ns.append(G * APL)
            for kind in ("flock", "tdm"):
                for i, N in enumerate(ns):
                    # per kernel: the default narrow ragged and full cases, and the huge narrow and wide ones, take
                    # different Flock bundles
                    bundle = "B" if (i == 1 or (build == "huge" and wide) or (build == "default" and wide)) else "A"
                    pile = PILE[(kind, "huge" if build == "huge" else ("wide" if wide else "narrow"))][N]
                    out.append(dict(build=build, G=G, APL=APL, kind=kind, wide=wide, N=N, bundle=bundle, pile=pile))
    return out


CASES = _cases()


def _case_id(c):
    return "%s-%s-G%d-APL%d-%s-N%d" % (c["build"], c["kind"], c["G"], c["APL"], "wide" if c["wide"] else "narrow", c["N"])


def _launch(c):
    """(threads per block, E, max_touching) of a case: E leaves the last block ragged."""
    N, pairs = c["N"], c["N"] * (c["N"] - 1) // 2
    if c["wide"]:
        threads = WIDE_THREADS[(c["build"], c["APL"])]
        per_block = threads // 32
    else:
        threads = 128
        per_block = 4 * (32 // c["G"])
    E = per_block + (3 if per_block > 8 else per_block // 2 + 1)
    if c["build"] == "huge":
        mt = pairs
    else:
        mt = DEFAULT_WIDE_TOUCHING[c["APL"]] if c["wide"] else min(pairs, 240)
    return threads, E, mt


def _flock_spawn(rng, E, N, T, pile):
    """Env e spawns in a square of side pile, 2.5 sqrt(N) m or the reference's 20 m, in turn."""
    pos = np.empty((E, N, 2))
    for e in range(E):
        side = (pile, 2.5 * np.sqrt(N), 20.0)[e % 3]
        pos[e] = side * (rng.random((N, 2)) - 0.5)
    ang = rng.uniform(-1, 1, (E, N)) * np.pi
    ta = 2 * np.pi * rng.random((E, T))
    td = 25 + rng.random((E, T)) * 35
    return pos, ang, np.stack([td * np.cos(ta), td * np.sin(ta)], -1)


def _tdm_spawn(rng, E, teams, pile):
    """combat.py's spawn in a pile arena, one twice as wide and the default 30 m one, in turn."""
    parts = [tdm_spawn(rng, 1, teams, *((pile, pile), (2 * pile, 2 * pile), (30.0, 30.0))[e % 3]) for e in range(E)]
    return parts[0][0], np.concatenate([p[1] for p in parts]), np.concatenate([p[2] for p in parts])


STEPS, CHUNK = 64, 16
OUTPUTS = ("obs", "nn_idx", "rewards", "collided", "done")


@pytest.fixture
def block_threads():
    """Set MACM_BLOCK_THREADS (read when a sim is created) for the test's sims; restored afterwards."""
    old = os.environ.get("MACM_BLOCK_THREADS")

    def set_(t):
        os.environ["MACM_BLOCK_THREADS"] = str(t)
    yield set_
    if old is None:
        os.environ.pop("MACM_BLOCK_THREADS", None)
    else:
        os.environ["MACM_BLOCK_THREADS"] = old


def _make(c, E, mt, rng):
    """Three sims of the case on the same spawn (stepped singly, by rollouts, by one-step rollouts) + the oracle."""
    import gym_macm
    from oracle import oracle
    N, pairs = c["N"], c["N"] * (c["N"] - 1) // 2
    if c["kind"] == "flock":
        kw = dict(FLOCK_A if c["bundle"] == "A" else FLOCK_B)
        targets = [i % 3 for i in range(N)] if (c["bundle"] == "B" and N >= 3) else None
        T = 1 if targets is None else 3
        pos, ang, tg = _flock_spawn(rng, E, N, T, c["pile"])
        sims = []
        for _ in range(3):
            s = gym_macm.BatchedFlock(E, n_agents=[N], targets=targets, device="cuda:0", seed=None,
                                      max_contacts=pairs, max_touching=mt, **kw)
            s.load_state(pos, ang, targets=tg)
            sims.append(s)
        ref = oracle.OracleBatch(E, n_agents=N, n_targets=T, **oracle_kwargs(kw))
        ref.reset(pos, ang, targets=tg, target_idx=targets)
        return sims, ref, kw
    teams = _teams(N)
    team, pos, ang = _tdm_spawn(rng, E, teams, c["pile"])
    sims = []
    for _ in range(3):
        s = gym_macm.BatchedTDM(E, n_agents=teams, device="cuda:0", seed=None, max_contacts=pairs, max_touching=mt)
        s.load_state(pos, ang)
        sims.append(s)
    ref = oracle.OracleBatch(E, env_kind=oracle.TDM, n_agents=N, n_targets=0)
    ref.reset(pos, ang, team=team)
    return sims, ref, {}


@pytest.mark.parametrize("c", CASES, ids=[_case_id(c) for c in CASES])
def test_kernel_against_oracle(c, block_threads):
    import torch
    threads, E, mt = _launch(c)
    block_threads(threads)
    G, APL, N = c["G"], c["APL"], c["N"]
    rng = np.random.default_rng(1000 * G + 10 * APL + N + (7 if c["kind"] == "tdm" else 0))
    (one, roll, step1), ref, kw = _make(c, E, mt, rng)
    for s in (one, roll, step1):
        info = s.engine.info
        assert (info.lanes_per_env, info.agents_per_lane, info.threads_per_block) == (G, APL, threads), _case_id(c)
        assert (s.engine.sizes.touch_scratch > 0) == (c["build"] == "huge"), _case_id(c)
    assert info.blocks == (E + info.envs_per_block - 1) // info.envs_per_block and E % info.envs_per_block, "ragged"
    flock = c["kind"] == "flock"
    cont = kw.get("action_mode") == "continuous"
    coord, rmode = kw.get("coord", "polar"), kw.get("reward_mode", "binary")
    attack_p = 0.9 if N % 2 else 0.5
    if flock:
        torch.cuda.synchronize()
        compare_obs(one.state["obs"].cpu().numpy(), ref.flock_observe(), coord)
    max_tc, max_ref_tc, deaths, per = 0, 0, 0, {}
    chunk = []
    for k in range(STEPS):
        if cont:
            a = rng.uniform(-1.2, 1.2, (E, N, 2)).astype(np.float32)
            act_t = torch.as_tensor(a, device="cuda:0")
            o = ref.flock_step(a.astype(np.float64))
        else:
            a = rng.integers(0, 3, (E, N, 4))
            if flock:
                a[..., 3] = 0
                o = ref.flock_step(a[..., :3])
            else:
                a[..., 3] = rng.random((E, N)) < attack_p
                o = ref.tdm_step(a)
            act_t = torch.as_tensor(a.astype(np.uint8), device="cuda:0")
        one.step(act_t)
        out1 = step1.rollout(act_t[None])    # one-step rollout with per-step outputs
        if flock:
            compare_step(one, ref, o, k, coord, rmode)
        else:
            deaths = int((~compare_tdm_step(one, ref, o, k, contact_envs=None)).sum())
        # the step's touching contacts; the device reports at most the shared stage's 240, the oracle all of them
        max_tc = max(max_tc, int(one.state["env_state"][:, 2].max()))
        max_ref_tc = max(max_ref_tc, max(ref.env_info(e)["touching"] for e in range(E)))
        chunk.append(act_t)
        for n in OUTPUTS:
            if n in one.state:
                per.setdefault(n, []).append(one.state[n].clone())
                assert torch.equal(step1.state[n], one.state[n]), "step %d: one-step rollout, %s" % (k, n)
                assert torch.equal(out1[n][0], one.state[n]), "step %d: one-step rollout output, %s" % (k, n)
        if len(chunk) == CHUNK:
            out = roll.rollout(torch.stack(chunk))
            torch.cuda.synchronize()
            for n in per:
                assert torch.equal(out[n], torch.stack(per[n])), "rollout up to step %d: %s" % (k, n)
            _same_state(one, roll, "rollout up to step %d" % k)
            chunk, per = [], {}
    _same_state(one, step1, "one-step rollouts")
    assert not chunk
    # the level-scheduled solver ran (more touching contacts than lanes), where N allows it
    if N * (N - 1) // 2 > G:
        assert max_tc > G, (max_tc, G)
    if c["build"] == "huge" and APL > 1:
        assert max_ref_tc > 240, max_ref_tc  # the global-memory stage held a pile
    if not flock and N >= 13:
        assert deaths > 0
    for s in (one, roll, step1):
        s.close()


def test_every_dispatched_kernel_has_a_case():
    """The cases cover DISPATCH_SHAPE x {default narrow; default wide, huge narrow, huge wide for G = 32}; a shape
    added without a case here fails."""
    expected = set()
    for kind in ("flock", "tdm"):
        for G, APL in ((4, 1), (8, 1), (16, 1), (32, 1), (32, 2), (32, 4)):
            expected.add(("default", G, APL, kind, False))
            if G == 32:
                expected |= {("default", G, APL, kind, True), ("huge", G, APL, kind, False), ("huge", G, APL, kind, True)}
    assert {(c["build"], c["G"], c["APL"], c["kind"], c["wide"]) for c in CASES} == expected
    assert len(expected) == 30
    # every kernel sees both Flock settings bundles
    for G, APL in SHAPES:
        for build in ("default", "huge"):
            got = {c["bundle"] for c in CASES if (c["build"], c["G"], c["APL"], c["kind"]) == (build, G, APL, "flock")}
            assert got in ({"A", "B"}, set()) and (got or build == "huge"), (build, G, APL)
