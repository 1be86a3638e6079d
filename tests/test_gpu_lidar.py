"""macm_lidar on the device against the oracle's scan (test_lidar_cpu.oracle_scan: the oracle's closest-hit ray cast
once per ray, which tests/test_lidar_cpu.py holds to a numpy restatement of the rule): stepped, gathered and piled
Flock batches at every dispatched agent count, TDM with dead agents, ray counts, fans and ranges across their limits,
worlds built against the cull's margins, env lists with repeats and bad device indices, 16-bit fractions, output
reuse, no host synchronisation, stream order, and a state that scanning leaves untouched.

Fraction bits and hit ids must be equal on every ray but the ambiguous ones: those where moving cos / sin of th by
2 ulp of float64 changes the fp32 dx or dy, because the device's float64 sin / cos and libm's may differ there."""
import ctypes as C
import math

import numpy as np
import pytest

from test_lidar_cpu import oracle_scan

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
f32 = np.float32


def ambiguous(ang, n_rays, fov, L):
    """bool [N,R]: rays whose fp32 dx or dy changes when cos / sin of th move by 2 ulp of float64."""
    r = np.arange(n_rays)
    o = fov * ((2 * r + 1 - n_rays).astype(np.float64) / float(2 * n_rays))
    th = np.asarray(ang, f32).astype(np.float64)[:, None] + o[None, :]
    amb = np.zeros(th.shape, bool)
    for fn in (np.cos, np.sin):
        v = fn(th)
        u = 2 * np.spacing(np.abs(v))
        base = (L * v).astype(f32)
        amb |= ((L * (v - u)).astype(f32) != base) | ((L * (v + u)).astype(f32) != base)
    return amb


class Worlds(object):
    """Env rows as fp32 positions [B,N,2], angles [B,N] and proxy bits [B,N]; `lidar` is the oracle's scan of each
    (test_lidar_cpu.oracle_scan: the oracle's closest-hit ray cast, once per ray)."""

    def __init__(self, pos, ang, proxy=None, radius=0.5):
        self.pos, self.ang = np.asarray(pos, f32), np.asarray(ang, f32)
        self.proxy = np.ones(self.ang.shape, bool) if proxy is None else np.asarray(proxy, bool)
        self.radius = float(radius)

    def lidar(self, n_rays, fov, L):
        rows = [oracle_scan(self.pos[b], self.ang[b], n_rays, fov, L, self.proxy[b], self.radius)
                for b in range(len(self.ang))]
        return np.stack([f for f, _ in rows]), np.stack([h for _, h in rows])


def oracle_of(env, envs=None):
    """The device's bodies (positions, angles; every Flock agent has a proxy) of `envs` (None: every env)."""
    st = env.state
    pos = st["posvel"][..., 0:2].cpu().numpy()
    ang = st["angsleep"][..., 0].cpu().numpy()
    if envs is not None:
        pos, ang = pos[list(envs)], ang[list(envs)]
    return Worlds(pos, ang, radius=env.settings.bodySettings["fixtures"].radius)


def check(env, ref, n_rays, fov, L, envs=None, fraction=None, hit=None, max_share=1e-5):
    """The device scan of env rows `envs` equals the oracle's scan of `ref` (a Worlds, one world per row) on every
    non-ambiguous ray; returns (rays compared, ambiguous rays, hits)."""
    import torch
    if fraction is None:
        fraction, hit = env.lidar(n_rays, L, fov, envs=envs)
    torch.cuda.synchronize()
    got_f = fraction.float().cpu().numpy()
    got_h = hit.cpu().numpy()
    want_f, want_h = ref.lidar(n_rays, fov, L)
    amb = np.stack([ambiguous(ref.ang[b], n_rays, fov, L) for b in range(len(ref.ang))])
    bad = ((got_f.view(np.int32) != want_f.view(np.int32)) | (got_h != want_h)) & ~amb
    assert not bad.any(), "%d rays differ, first (row, agent, ray) %s: device (%r, %d), oracle (%r, %d)" % (
        bad.sum(), np.argwhere(bad)[0], got_f[bad][0], got_h[bad][0], want_f[bad][0], want_h[bad][0])
    assert amb.sum() <= max(2, max_share * amb.size), "%d of %d rays ambiguous" % (amb.sum(), amb.size)
    return amb.size, int(amb.sum()), int((want_h >= 0).sum())


def _flock(E, N, T=1, steps=20, seed=1, spread=None, policy="flock", **kw):
    import torch
    import gym_macm
    spread = spread if spread is not None else max(3.0, 1.5 * np.sqrt(N))
    env = gym_macm.BatchedFlock(E, n_agents=[N], targets=[i % T for i in range(N)], device=DEV, seed=seed,
                                start_spread=spread, **kw)
    for k in range(steps):
        env.step(env.bot_actions(policy if k % 3 else "random", seed=k))
    torch.cuda.synchronize()
    return env


def _loaded(pos, ang, **kw):
    """A Flock batch holding the given worlds [E,N,2] / [E,N]."""
    import gym_macm
    E, N = np.shape(ang)
    env = gym_macm.BatchedFlock(E, n_agents=[N], device=DEV, seed=None, **kw)
    env.load_state(np.asarray(pos, np.float64), np.asarray(ang, np.float64), targets=np.zeros((E, 1, 2)))
    return env


@pytest.mark.parametrize("N", [2, 4, 6, 16, 32, 33, 64, 65, 100, 128])
def test_flock_against_the_oracle(N):
    env = _flock(6, N, T=min(N, 4), steps=25, seed=N)
    total = [0, 0, 0]
    for R, fov, L in ((32, 2 * np.pi, 10.0), (33, np.pi, 1.0), (3, 0.3, 1e4), (1, 2 * np.pi, 0.01)):
        for k, v in enumerate(check(env, oracle_of(env), R, fov, L)):
            total[k] += v
    assert total[2] > 0
    print("N=%d: %d rays, %d ambiguous, %d hits" % (N, *total))


def test_gathered_flock_and_spawn_pile():
    # a flock gathered at its target by the device `flock` actor, and a pile of overlapping discs
    env = _flock(8, 64, T=1, steps=300, seed=3, spread=12.0)
    for R, fov, L in ((32, 2 * np.pi, 10.0), (1024, 2 * np.pi, 10.0), (128, np.pi, 1.0)):
        check(env, oracle_of(env), R, fov, L)
    rng = np.random.default_rng(4)
    pile = _loaded(rng.uniform(-0.8, 0.8, (4, 40, 2)), rng.uniform(-np.pi, np.pi, (4, 40)))
    for R, fov, L in ((32, 2 * np.pi, 10.0), (33, 0.3, 0.01), (1024, 2 * np.pi, 1.0)):
        check(pile, oracle_of(pile), R, fov, L)


def test_tdm_with_dead_agents():
    import torch
    import gym_macm
    from oracle import oracle
    rng = np.random.default_rng(5)
    E, teams = 12, [6, 6, 6]
    team = np.repeat(np.arange(3), 6).astype(np.uint8)
    N = len(team)
    pos = np.stack([rng.random((E, N)) * (team[None] + 3.0), rng.random((E, N)) * 6.0], -1)
    ang = rng.uniform(-1, 1, (E, N)) * np.pi
    env = gym_macm.BatchedTDM(E, n_agents=teams, device=DEV, seed=None, max_contacts=N * (N - 1) // 2,
                              max_touching=N * (N - 1) // 2)
    env.load_state(pos, ang)
    ref = oracle.OracleBatch(E, env_kind=oracle.TDM, n_agents=N, n_targets=0)
    ref.reset(pos, ang, team=team)
    for _ in range(300):
        act = np.concatenate([rng.integers(0, 3, (E, N, 3)), (rng.random((E, N, 1)) < 0.9).astype(np.int64)], -1)
        env.step(torch.as_tensor(act, device=DEV))
        ref.tdm_step(act)
    torch.cuda.synchronize()
    st = env.state
    assert np.array_equal(st["posvel"].cpu().numpy()[..., 0:2], ref.bodies()[..., 0:2])
    alive = ref.tdm_state()[..., 3] > 0
    assert np.array_equal(env.alive.cpu().numpy(), alive) and (~alive).sum() > E
    worlds = Worlds(ref.bodies()[..., 0:2], ref.bodies()[..., 4], alive)
    for R, fov, L in ((32, 2 * np.pi, 10.0), (33, np.pi, 4.0)):
        check(env, worlds, R, fov, L)
    _, hit = env.lidar(64, 10.0)
    h = hit.cpu().numpy()
    dead_ids = [set(np.flatnonzero(~alive[e])) for e in range(E)]
    assert not any(set(h[e].ravel()) & dead_ids[e] for e in range(E)), "a ray reported a dead agent"


def test_cull_adversarial_worlds():
    """Bodies tangent to rays, at fraction 1, in gaps between two discs, an agent 1 km away, and reaches so large that
    every body is a candidate: the cull must keep every body the exact test can hit."""
    rng = np.random.default_rng(6)
    E, N, R, fov, L = 16, 24, 32, 2 * np.pi, 4.0
    pos = np.zeros((E, N, 2))
    ang = rng.uniform(-np.pi, np.pi, (E, N))
    for e in range(E):
        a = float(f32(ang[e, 0]))
        for j in range(1, N):
            r = int(rng.integers(R))
            th = a + fov * ((2 * r + 1 - R) / (2 * R))
            u, n = np.array([np.cos(th), np.sin(th)]), np.array([-np.sin(th), np.cos(th)])
            kind = j % 4
            if kind == 0:     # tangent, to within rounding, on either side
                c = rng.uniform(1.0, L) * u + (0.5 + rng.choice([-1, 0, 1]) * rng.uniform(0, 3e-7)) * n
            elif kind == 1:   # at fraction 1, to within rounding
                c = (L + 0.5 + rng.uniform(-3e-7, 3e-7)) * u
            elif kind == 2:   # one disc of a grazing pair: the ray runs through the gap
                c = rng.uniform(1.0, L) * u + (0.5 + rng.uniform(0, 1e-6)) * n * (1 if j % 8 == 2 else -1)
            else:
                c = rng.uniform(-L, L, 2)
            pos[e, j] = c
        pos[e, N - 1] = (1000.0, -1000.0)   # far away
    env = _loaded(pos, ang)
    n_amb, n_hits = 0, 0
    for RR, fv, LL in ((R, fov, L), (R, fov, 1e4), (1024, 2 * np.pi, 1e6), (7, 1e-3, L)):
        _, a, h = check(env, oracle_of(env), RR, fv, LL, max_share=1e-3)
        n_amb += a
        n_hits += h
    assert n_hits > E * N
    # every agent far from the origin: rounding of p2 large against a short reach
    far = _loaded(pos + 3000.0, ang)
    for RR, LL in ((32, 0.01), (32, 2.0), (1024, 1.0)):
        check(far, oracle_of(far), RR, 2 * np.pi, LL, max_share=1e-3)


def test_env_subsets_and_bad_device_indices():
    import torch
    from gym_macm import _lib
    env = _flock(5, 16, T=2, steps=15, seed=7)
    envs = [3, 0, 3, 4, 1]
    check(env, oracle_of(env, envs), 32, 2 * np.pi, 10.0, envs=envs)
    f_list, h_list = env.lidar(32, 10.0, envs=envs)
    f_ten, h_ten = env.lidar(32, 10.0, envs=torch.tensor(envs, device=DEV))
    assert torch.equal(f_list, f_ten) and torch.equal(h_list, h_ten)
    for kw in (dict(envs=[0, 5]), dict(envs=[-1])):
        with pytest.raises(ValueError):
            env.lidar(32, 10.0, **kw)
    # the same indices straight to the ABI: rows of misses, nothing read out of bounds
    bad = torch.tensor([-1, 5, 1 << 30, -(1 << 31), 2], dtype=torch.int32, device=DEV)
    fr = torch.full((5, 16, 33), 7.0, device=DEV)
    hit = torch.full((5, 16, 33), 7, dtype=torch.int32, device=DEV)
    a = _lib.MacmLidarArgs(5, 33, 10.0, math.pi, bad.data_ptr(), fr.data_ptr(), hit.data_ptr())
    assert _lib.lib().macm_lidar(env.engine._h, C.byref(a), None) == 0
    torch.cuda.synchronize()
    assert (fr[:4] == 1).all() and (hit[:4] == -1).all()
    check(env, oracle_of(env, [2]), 33, math.pi, 10.0, fraction=fr[4:], hit=hit[4:])


def test_abi_errors():
    import torch
    from gym_macm import _lib
    L = _lib.lib()
    env = _flock(4, 8, steps=2)
    fr = torch.zeros((6, 8, 16), device=DEV)
    hit = torch.zeros((6, 8, 16), dtype=torch.int32, device=DEV)

    def call(n=4, R=16, rng=5.0, fov=1.0, envs=None, f=fr.data_ptr(), h=hit.data_ptr(), handle=env.engine._h):
        a = _lib.MacmLidarArgs(n, R, rng, fov, envs, f, h)
        return L.macm_lidar(handle, C.byref(a), None)

    assert call() == 0 and call(h=None) == 0
    for bad in (dict(n=0), dict(n=5), dict(R=0), dict(R=1025), dict(rng=0.0), dict(rng=-1.0), dict(rng=1e6 * 1.01),
                dict(rng=float("inf")), dict(rng=float("nan")), dict(fov=0.0), dict(fov=2 * math.pi + 1e-12),
                dict(fov=float("nan")), dict(f=None)):
        assert call(**bad) == -1, bad                            # MACM_E_INVALID
    idx = torch.zeros(8, dtype=torch.int32, device=DEV)
    assert call(n=2, envs=idx.data_ptr() + 2) == -4              # MACM_E_ALIGN
    assert call(h=hit.data_ptr() + 2) == -4
    assert call(f=fr.data_ptr() + 2) == -4
    p = _lib.default_params(_lib.FLOCK)
    unbound = C.c_void_p()
    assert L.macm_create(C.byref(unbound), C.byref(p), 0) == 0
    try:
        assert call(handle=unbound) == -3                        # MACM_E_UNBOUND
    finally:
        L.macm_destroy(unbound)


@pytest.mark.parametrize("dtype", ["float16", "bfloat16"])
def test_16bit_fractions_are_the_rounded_fp32_scan(dtype):
    import torch
    # the `flock` actor reads the stored observation, so it refuses a 16-bit one: both twins walk randomly
    a = _flock(6, 32, T=2, steps=20, seed=8, policy="random")
    b = _flock(6, 32, T=2, steps=20, seed=8, policy="random", obs_dtype=dtype)
    for R, L in ((32, 10.0), (33, 1.0)):
        fa, ha = a.lidar(R, L)
        fb, hb = b.lidar(R, L)
        torch.cuda.synchronize()
        assert fb.dtype == getattr(torch, dtype) and torch.equal(ha, hb)
        assert torch.equal(fb.view(torch.int16), fa.to(fb.dtype).view(torch.int16))


def test_hits_false_out_reuse_and_no_host_sync():
    import torch
    env = _flock(8, 64, T=2, steps=10, seed=9)
    f, h = env.lidar(32, 10.0)
    f2, h2 = env.lidar(32, 10.0, hits=False)
    assert h2 is None and torch.equal(f, f2)
    out = (torch.full_like(f, 5.0), torch.full_like(h, 5))
    torch.cuda.set_sync_debug_mode("error")
    try:
        r = env.lidar(32, 10.0, out=out)
        env.lidar(32, 10.0, out=(torch.empty_like(f), None), hits=False)
        env.lidar(128, 3.0, fov=1.0)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert r[0] is out[0] and r[1] is out[1]
    check(env, oracle_of(env), 32, 2 * np.pi, 10.0, fraction=out[0], hit=out[1])
    for o in ((f.cpu(), h), (f.double(), h), (f, h.long()), (f[:, :, :16], h), (f, None)):
        with pytest.raises(ValueError):
            env.lidar(32, 10.0, out=o)


def test_stream_order_and_batch_pool():
    import torch
    import gym_macm
    E, N = 8, 16
    s = torch.cuda.Stream(device=DEV)
    env = gym_macm.BatchedFlock(E, n_agents=[N], device=DEV, seed=9, start_spread=5.0, stream=s)
    acts = [torch.randint(0, 3, (E, N, 3), device=DEV) for _ in range(6)]
    s.wait_stream(torch.cuda.current_stream(DEV))
    for a in acts:
        env.step(a)
    f, h = env.lidar(32, 6.0)      # right after the steps, on the batch's stream, no sync in between
    s.synchronize()
    check(env, oracle_of(env), 32, 2 * np.pi, 6.0, fraction=f, hit=h)

    pool = gym_macm.BatchPool([gym_macm.BatchedFlock(E, n_agents=[N], device=DEV, seed=20 + r, start_spread=5.0)
                               for r in range(2)])
    packed = [pool.batches[0].pack_actions(a).clone() for a in acts]
    torch.cuda.synchronize()
    last = {}
    for k, a in enumerate(packed):
        b = pool.step(a)
        last[k % 2] = (b, b.lidar(32, 6.0))
    pool.synchronize()
    for b, (f, h) in last.values():
        check(b, oracle_of(b), 32, 2 * np.pi, 6.0, fraction=f, hit=h)


def test_scanning_leaves_the_state_untouched():
    import torch
    a, b = _flock(8, 32, T=2, steps=12, seed=5), _flock(8, 32, T=2, steps=12, seed=5)
    before = {n: t.clone() for n, t in a.engine.t.items()}
    launches = a.engine.launch_count
    a.lidar(64, 10.0)
    torch.cuda.synchronize()
    assert a.engine.launch_count == launches + 1
    for n, t in a.engine.t.items():
        assert torch.equal(t, before[n]), n
    for k in range(5):
        acts = torch.randint(0, 3, (8, 32, 3), device=DEV)
        a.lidar(32, 5.0)
        a.step(acts)
        b.step(acts)
    torch.cuda.synchronize()
    for n in a.engine.t:
        assert torch.equal(a.engine.t[n], b.engine.t[n]), n
