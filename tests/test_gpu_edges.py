"""Predicates of the step at their exact edges, against the oracle.

The kernel takes several decisions on fp32 values that were chosen to reproduce the reference's float64 or Box2D
decisions: the binary reward threshold, touching, fat-AABB overlap, nearest-agent draws and the TDM ray cast.
Random states essentially never land on their boundaries, so each test here places agents so that the quantity
the predicate sees is exactly on the boundary, or one fp32 ulp to either side.  Agents are idle and at rest, so the
loaded positions are the ones the predicates see, step after step.
"""
import os

import numpy as np
import pytest

from _parity import compare_obs, compare_step
from test_gpu_tdm import compare_tdm_step

pytestmark = pytest.mark.gpu

f32 = np.float32


def _prev(x):
    return np.nextafter(f32(x), f32(-np.inf))


def _next(x):
    return np.nextafter(f32(x), f32(np.inf))


def _d2(ax, ay, bx, by):
    """b2DistanceSquared of the kernel in fp32, no FMA: dx = b.x - a.x; dx * dx + dy * dy."""
    dx, dy = f32(bx) - f32(ax), f32(by) - f32(ay)
    return dx * dx + dy * dy


def _place_at_d2(ax, ay, r, want, K=1200):
    """An fp32 point b near a + r (0.6, -0.8) whose _d2(a, b) is exactly `want` (numpy's fp32 arithmetic rounds each
    operation like the kernel, which is built without FMA contraction)."""
    ax, ay = f32(ax), f32(ay)
    off = np.arange(-K, K, dtype=np.int32)
    bx = (np.array([ax + f32(0.6 * r)], f32).view(np.int32) + off).view(f32)
    by = (np.array([ay - f32(0.8 * r)], f32).view(np.int32) + off).view(f32)
    dx, dy = bx - ax, by - ay
    d2 = dx[:, None] * dx[:, None] + dy[None, :] * dy[None, :]
    hit = np.argwhere(d2 == f32(want))
    assert len(hit), "no fp32 point at d2 = %r" % want
    i, j = hit[len(hit) // 2]
    assert _d2(ax, ay, bx[i], by[j]) == f32(want)
    return bx[i], by[j]


def _flock(E, N, pos, targets, **kw):
    import torch
    import gym_macm
    from oracle import oracle
    from _parity import oracle_kwargs
    env = gym_macm.BatchedFlock(E, n_agents=[N], device="cuda:0", seed=None, **kw)
    env.load_state(pos, np.zeros((E, N)), targets=targets)
    ref = oracle.OracleBatch(E, n_agents=N, n_targets=1, **oracle_kwargs(kw))
    ref.reset(pos, np.zeros((E, N)), targets=targets)
    torch.cuda.synchronize()
    return env, ref


def _idle_steps(env, ref, n=2, coord="polar", reward_mode="binary"):
    import torch
    E, N = ref.E, ref.N
    idle = np.ones((E, N, 3), np.int64)
    for k in range(n):
        env.step(torch.as_tensor(idle, device="cuda:0"))
        o = ref.flock_step(idle)
        compare_step(env, ref, o, k, coord, reward_mode)
    return o


def _far(E, N, x0=300.0):
    """Positions of agents that take no part: on a line far from the target and from each other (no contacts)."""
    pos = np.zeros((E, N, 2))
    pos[:, :, 0] = x0 + 3.0 * np.arange(N)
    pos[:, :, 1] = -200.0
    return pos


@pytest.mark.parametrize("R", [7.0, 0.5, 2.5, 3.3, 10.1])
def test_binary_reward_threshold(R):
    """reward = int(sqrt64(d2) < R) is folded into d2 < thr with an fp32 thr; agents at d2 = prev(thr), thr and
    next(thr) from their target get 1, 0, 0 -- on the device, in the oracle and in a float64 restatement."""
    import gym_macm
    probe = gym_macm.BatchedFlock(1, n_agents=[2], device="cuda:0", seed=None, _reward_radius=R)
    thr = f32(probe.engine.info.binary_d2_threshold)
    probe.close()
    assert np.sqrt(np.float64(_prev(thr))) < R and not np.sqrt(np.float64(thr)) < R, (R, thr)
    tx, ty = f32(47.3), f32(-31.9)      # away from the origin, so the subtraction rounds
    E, N = 3, 4
    pos = _far(E, N)
    want = (_prev(thr), thr, _next(thr))
    for e in range(E):
        pos[e, 0] = _place_at_d2(tx, ty, R, want[e])
    targets = np.tile(np.array([tx, ty], np.float64), (E, 1, 1))
    env, ref = _flock(E, N, pos, targets, _reward_radius=R)
    o = _idle_steps(env, ref)
    rew = env.state["rewards"].cpu().numpy()
    d64 = [np.sqrt(np.float64(_d2(tx, ty, *pos[e, 0]))) for e in range(E)]
    expect = [float(d < R) for d in d64]          # the reference's test, in float64 on the fp32 d2
    assert expect == [1.0, 0.0, 0.0]
    assert list(rew[:, 0]) == expect and list(o["rewards"][:, 0]) == expect
    env.close()


def test_touching_at_rsum2():
    """Touching is !(d2 > rsum2): a pair exactly at d2 = rsum2 = 1 touches, one ulp inside touches, one ulp outside
    is listed (fat AABBs overlap) but does not touch."""
    E, N = 3, 4
    pos = _far(E, N)
    ax, ay = f32(13.7), f32(-5.3)
    rsum2 = f32(1.0)
    for e, want in enumerate((rsum2, _prev(rsum2), _next(rsum2))):
        pos[e, 0] = (ax, ay)
        pos[e, 1] = _place_at_d2(ax, ay, 1.0, want)
    tg = np.tile(np.array([40.0, 40.0]), (E, 1, 1))
    env, ref = _flock(E, N, pos, tg)
    for k in range(2):
        _idle_steps(env, ref, 1)
        for e, touching in enumerate((1, 1, 0)):
            ab, fl, imp = env.contacts(e)
            assert ab.tolist() == [[0, 1]] and fl.tolist() == [touching], (k, e, ab, fl)
    assert env.state["collided"][:, :2].all()
    env.close()


def test_fat_aabbs_that_abut():
    """b2TestOverlap counts equality as overlap: fat AABBs that share an edge give a listed, non-touching contact
    (reward -1 for both agents, reference defect B1); one ulp apart, no contact."""
    E, N = 4, 4
    pos = _far(E, N)
    r, ext = f32(0.5), f32(0.1)
    a = (f32(-7.9), f32(-12.6))   # (at 3.3, (c - r) - ext skips every other fp32 value near 3.9: no exact abutment)
    for e in range(E):
        axis = e // 2
        hi = (a[axis] + r) + ext                            # agent 0's fat upper bound on the axis
        want = hi if e % 2 == 0 else _next(hi)              # agent 1's fat lower bound
        c = (np.array([a[axis] + f32(1.2)], f32).view(np.int32) + np.arange(-64, 64, dtype=np.int32)).view(f32)
        lo = (c - r) - ext
        j = np.flatnonzero(lo == want)
        assert len(j), (e, want)
        b = list(a)
        b[axis] = c[j[0]]
        pos[e, 0], pos[e, 1] = a, b
    tg = np.tile(np.array([40.0, 40.0]), (E, 1, 1))
    env, ref = _flock(E, N, pos, tg)
    fat = env.state["fat"].cpu().numpy()
    for e in range(E):
        axis = e // 2
        gap = fat[e, 1, axis] - fat[e, 0, 2 + axis]
        assert gap == 0 if e % 2 == 0 else gap > 0
    for k in range(2):
        _idle_steps(env, ref, 1)
        for e in range(E):
            ab, fl, _ = env.contacts(e)
            if e % 2 == 0:
                assert ab.tolist() == [[0, 1]] and fl.tolist() == [0], (e, ab, fl)
            else:
                assert len(ab) == 0, (e, ab)
    rew = env.state["rewards"].cpu().numpy()
    assert (rew[0::2, :2] == -1).all() and (rew[1::2, :2] != -1).all()
    env.close()


@pytest.fixture
def block_threads():
    old = os.environ.get("MACM_BLOCK_THREADS")

    def set_(t):
        os.environ["MACM_BLOCK_THREADS"] = str(t)
    yield set_
    if old is None:
        os.environ.pop("MACM_BLOCK_THREADS", None)
    else:
        os.environ["MACM_BLOCK_THREADS"] = old


@pytest.mark.parametrize("threads", [128, 448])
@pytest.mark.parametrize("N,cols", [(65, 9), (100, 10), (128, 11)])
def test_nn_exact_draws_four_agents_per_lane(N, cols, threads, block_threads):
    """Agents on a 2 m lattice in shuffled index order: most have two to four nearest neighbours at exactly the same
    distance, and the lowest index must win (mvmnt.py:194).  Four agents per lane search in blocks of four
    candidates (strict '<' between blocks, lowest index inside the winning one)."""
    import torch
    import gym_macm
    from oracle import oracle
    block_threads(threads)
    E = 4
    rng = np.random.default_rng(N)
    idx = np.arange(N)
    base = np.stack([2.0 * (idx % cols), 2.0 * (idx // cols)], -1)
    pos = np.stack([base[rng.permutation(N)] + off for off in ((0, 0), (-7, 3), (100, -50), (0.5, 0.25))])
    ang = rng.uniform(-3, 3, (E, N))
    tg = rng.uniform(-40, 40, (E, 1, 2))
    env = gym_macm.BatchedFlock(E, n_agents=[N], device="cuda:0", seed=None)
    assert (env.engine.info.agents_per_lane, env.engine.info.threads_per_block) == (4, threads)
    env.load_state(pos, ang, targets=tg)
    ref = oracle.OracleBatch(E, n_agents=N, n_targets=1)
    ref.reset(pos, ang, targets=tg)
    idle = np.ones((E, N, 3), np.int64)
    draws = 0
    for k in range(2):
        env.step(torch.as_tensor(idle, device="cuda:0"))
        o = ref.flock_step(idle)
        torch.cuda.synchronize()
        got = env.state["nn_idx"].cpu().numpy()
        assert np.array_equal(got, o["nn_idx"]), "step %d" % k
        compare_obs(env.state["obs"].cpu().numpy(), o, "polar", k)
    # the draws are real: count agents whose nearest distance is shared by a higher index
    p = pos[0]
    d2 = ((p[:, None] - p[None]) ** 2).sum(-1) + np.eye(N) * 1e9
    draws = int(((d2 == d2.min(1, keepdims=True)).sum(1) > 1).sum())
    assert draws > N // 2
    env.close()


def _raycast_f32(p1, p2, c, radius=f32(0.5)):
    """b2CircleShape::RayCast in fp32 (the kernel's and Box2D's operation order): the fraction, or None."""
    p1, p2, c = [np.asarray(v, f32) for v in (p1, p2, c)]
    s = p1 - c
    b = (s[0] * s[0] + s[1] * s[1]) - radius * radius
    r = p2 - p1
    cq = s[0] * r[0] + s[1] * r[1]
    rr = r[0] * r[0] + r[1] * r[1]
    sigma = cq * cq - rr * b
    if sigma < 0 or rr < f32(1.1920929e-07):
        return None
    a = -(cq + np.sqrt(sigma))
    return a / rr if f32(0) <= a <= rr else None


def _hit64(p1, c, R=0.5, reach=2.0):
    """The geometry in float64: the segment p1 + t (reach, 0), t in [0, 1], meets the circle (not from inside)."""
    dx, dy = c[0] - p1[0], c[1] - p1[1]
    if dx * dx + dy * dy < R * R or abs(dy) > R:
        return None
    t = (dx - np.sqrt(R * R - dy * dy)) / reach
    return t if 0 <= t <= 1 else None


def _tdm(E, teams, pos, ang):
    import gym_macm
    from oracle import oracle
    N = sum(teams)
    team = np.array([t for t, n in enumerate(teams) for _ in range(n)], np.uint8)
    env = gym_macm.BatchedTDM(E, n_agents=teams, device="cuda:0", seed=None)
    env.load_state(pos, ang)
    ref = oracle.OracleBatch(E, env_kind=oracle.TDM, n_agents=N, n_targets=0)
    ref.reset(pos, ang, team=team)
    return env, ref


def _tdm_step(env, ref, attackers, k):
    """One step with everyone idle but `attackers` [(env, agent)], who attack."""
    import torch
    a = np.ones((ref.E, ref.N, 4), np.int64)
    a[..., 3] = 0
    for e, i in attackers:
        a[e, i, 3] = 1
    env.step(torch.as_tensor(a.astype(np.uint8), device="cuda:0"))
    o = ref.tdm_step(a)
    compare_tdm_step(env, ref, o, k, contact_envs=None)
    return env.health.cpu().numpy(), env.alive.cpu().numpy()


@pytest.mark.parametrize("pair", [(31, 32), (63, 64), (5, 100), (7, 39), (2, 98)])
def test_ray_cast_ties_across_lanes_and_slots(pair):
    """Two victims at exactly the same fraction of the attacker's ray (mirror images across it): the lower index
    is hit, whichever lane and slot each sits in -- agent i sits in lane i % 32, slot i // 32, so the pairs are
    split across lanes and slots, and (7, 39), (2, 98) share a lane."""
    lo, hi = pair
    N = hi + 2
    teams = [N // 2, N - N // 2]
    E = 2
    pos = np.zeros((E, N, 2))
    pos[:, :, 0] = 200.0 + 3.0 * np.arange(N)       # bystanders far away, apart
    pos[:, :, 1] = 150.0
    ang = np.zeros((E, N))
    atk = 0 if lo != 0 else N - 1
    p1 = (f32(10.0), f32(20.0))
    for e, (h, d) in enumerate(((0.3, 1.25), (0.45, 1.5))):
        pos[e, atk] = p1
        pos[e, lo] = (p1[0] + f32(d), p1[1] + f32(h))
        pos[e, hi] = (p1[0] + f32(d), p1[1] - f32(h))
        p2 = (p1[0] + f32(2.0), p1[1])
        fl, fh = _raycast_f32(p1, p2, pos[e, lo]), _raycast_f32(p1, p2, pos[e, hi])
        assert fl is not None and fl == fh
        assert _hit64(p1, pos[e, lo]) == _hit64(p1, pos[e, hi]) is not None
    env, ref = _tdm(E, teams, pos, ang)
    health, alive = _tdm_step(env, ref, [(e, atk) for e in range(E)], 0)
    for e in range(E):
        assert health[e, lo] == 0.75 and health[e, hi] == 1.0, (e, health[e, lo], health[e, hi])
    assert alive.all()
    env.close()


def test_ray_cast_end_and_origin():
    """The ray ends exactly on a victim's circle (fraction 1: a hit) or one ulp short of it (a miss); a ray whose
    origin lies inside another agent does not hit that agent; a dead agent in front of a live one does not shield it."""
    E, teams = 4, [5, 5]
    N = sum(teams)
    pos = np.zeros((E, N, 2))
    pos[:, :, 0] = 200.0 + 3.0 * np.arange(N)
    pos[:, :, 1] = 150.0
    ang = np.zeros((E, N))
    p1 = (f32(10.0), f32(20.0))
    reach = f32(2.0)
    # env 0: victim 6 at melee_range + radius; env 1: one ulp beyond
    for e, cx in ((0, p1[0] + reach + f32(0.5)), (1, _next(p1[0] + reach + f32(0.5)))):
        pos[e, 0], pos[e, 6] = p1, (cx, p1[1])
        hit = _raycast_f32(p1, (p1[0] + reach, p1[1]), pos[e, 6])
        assert (hit == 1.0) if e == 0 else (hit is None), (e, hit)
        assert (_hit64(p1, pos[e, 6]) == 1.0) if e == 0 else (_hit64(p1, pos[e, 6]) is None)
    # env 2: the attacker's origin lies inside agent 7 (centres 0.3 apart), nothing else on the ray
    pos[2, 0], pos[2, 7] = p1, (p1[0] + f32(0.3), p1[1])
    assert _raycast_f32(p1, (p1[0] + reach, p1[1]), pos[2, 7]) is None and _hit64(p1, pos[2, 7]) is None
    # env 3: agent 6 is killed by four attackers in step 0; in step 1 agent 0's ray passes where 6 was and hits 7
    D, L = (f32(9.4), f32(10.0)), (f32(10.65), f32(10.0))
    pos[3, 0], pos[3, 6], pos[3, 7] = (f32(8.3), f32(10.0)), D, L
    killers = {1: ((9.4, 11.4), -np.pi / 2), 2: ((9.4, 8.6), np.pi / 2), 3: ((10.4, 11.0), -3 * np.pi / 4),
               4: ((8.4, 11.0), -np.pi / 4)}
    for i, (p, a) in killers.items():
        pos[3, i], ang[3, i] = p, a
    env, ref = _tdm(E, teams, pos, ang)
    health, alive = _tdm_step(env, ref, [(0, 0), (1, 0), (2, 0)] + [(3, i) for i in killers], 0)
    assert health[0, 6] == 0.75 and health[1, 6] == 1.0
    assert health[2, 7] == 1.0
    assert not alive[3, 6] and health[3, 7] == 1.0
    health, alive = _tdm_step(env, ref, [(3, 0)], 1)
    assert health[3, 7] == 0.75
    env.close()
