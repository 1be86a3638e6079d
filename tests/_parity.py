"""Shared harness of the GPU parity tests: load identical states into the CUDA simulator (through
the C ABI) and into the CPU oracle, step both with the same actions, compare.

Bars (BASELINE.json north_star): contact (broadphase pair) sets, collision flags, nearest-agent
ids and binary rewards bit-exact; positions, velocities, fat AABBs, sleep timers and warm-start
impulses are ALSO bit-exact here because the kernel reproduces Box2D's fp32 operation order;
linear rewards and observation floats, which the reference computes in float64 and the kernel
in fp32, within OBS_RTOL / OBS_ATOL (angles compared modulo 2 pi).
"""
import numpy as np

OBS_RTOL, OBS_ATOL = 1e-5, 2e-6      # fp32 sqrt/atan2 against the oracle's float64
LIN_REWARD_ATOL = 1e-6               # 1 - d/35 with d <= ~100: a few fp32 ulps


def random_state(rng, E, N, T, spread=20.0):
    """The reference's initial distributions (mvmnt.py:48-52,62-64), as float64 draws."""
    pos = spread * (rng.random((E, N, 2)) - 0.5)
    ang = rng.uniform(-1, 1, (E, N)) * np.pi
    ta = 2 * np.pi * rng.random((E, T))
    td = 25 + rng.random((E, T)) * 35
    tg = np.stack([td * np.cos(ta), td * np.sin(ta)], -1)
    return pos, ang, tg


def gpu_bodies(env):
    st = env.state
    return np.concatenate([st["posvel"].cpu().numpy(), st["angsleep"].cpu().numpy(), st["fat"].cpu().numpy()], -1)


def ang_diff(a, b):
    d = np.abs(a - b) % (2 * np.pi)
    return np.minimum(d, 2 * np.pi - d)


def compare_step(env, ref, o, k, coord="polar", reward_mode="binary", check_contacts_envs=None):
    import torch
    torch.cuda.synchronize()
    E, N = ref.E, ref.N
    st = env.state
    assert not (st["env_state"][:, 1].cpu().numpy() & 6).any(), "step %d: contact capacity overflow" % k
    gb, rb = gpu_bodies(env), ref.bodies()
    names = ["x", "y", "vx", "vy", "angle", "sleep", "fat_lx", "fat_ly", "fat_hx", "fat_hy"]
    for c, nm in enumerate(names):
        bad = np.argwhere(gb[..., c] != rb[..., c])
        assert len(bad) == 0, "step %d: %s differs at %d agents, first (env,agent)=%s gpu=%r oracle=%r" % (
            k, nm, len(bad), bad[0], gb[tuple(bad[0])][c], rb[tuple(bad[0])][c])
    st = env.state
    assert np.array_equal(st["collided"].cpu().numpy(), o["collided"]), "step %d: collision flags" % k
    assert np.array_equal(st["nn_idx"].cpu().numpy(), o["nn_idx"]), "step %d: nearest-agent ids" % k
    assert np.array_equal(st["done"].cpu().numpy(), o["done"]), "step %d: done" % k
    rew = st["rewards"].cpu().numpy().astype(np.float64)
    if reward_mode == "binary":
        assert np.array_equal(rew, o["rewards"]), "step %d: binary rewards" % k
    else:
        assert np.array_equal(rew == -1, o["rewards"] == -1)
        assert np.allclose(rew, o["rewards"], rtol=0, atol=LIN_REWARD_ATOL), "step %d: linear rewards" % k
    # contact lists: same pairs in the same (birth) order, same touching flags, same impulses
    cnt = st["contact_count"].cpu().numpy()
    envs = range(E) if check_contacts_envs is None else check_contacts_envs
    for e in envs:
        ab, fl, imp = env.contacts(e)
        rab, rfl, rimp = ref.contacts(e)
        assert cnt[e] == len(rab), "step %d env %d: %d contacts vs oracle %d" % (k, e, cnt[e], len(rab))
        assert np.array_equal(ab, rab), "step %d env %d: contact pairs/order" % (k, e)
        assert np.array_equal(fl, rfl), "step %d env %d: touching flags" % (k, e)
        t = rfl.astype(bool)
        assert np.array_equal(imp[t], rimp[t]), "step %d env %d: warm-start impulses" % (k, e)
    compare_obs(st["obs"].cpu().numpy(), o, coord, k)


def compare_obs(obs, o, coord, k=0):
    D = obs.shape[-1] // 2
    nn, tg = obs[..., 0:D].astype(np.float64), obs[..., D:2 * D].astype(np.float64)
    for got, want, nm in ((nn, o["nn_pos"], "nn"), (tg, o["tg_pos"], "target")):
        assert np.allclose(got[..., 0], want[..., 0], rtol=OBS_RTOL, atol=OBS_ATOL), "step %d: %s distance" % (k, nm)
        if coord == "polar":
            assert ang_diff(got[..., 1], want[..., 1]).max() <= 2e-6 + 1e-6, "step %d: %s angle" % (k, nm)
        else:
            assert np.allclose(got[..., 1:3], want[..., 1:3], rtol=0, atol=3e-6), "step %d: %s cos/sin" % (k, nm)


def make_pair(E, N, targets=None, seed=0, spread=20.0, max_contacts=0, max_touching=0, **kw):
    """(BatchedFlock on cuda:0, OracleBatch) holding the same fresh worlds."""
    import gym_macm
    from oracle import oracle
    rng = np.random.default_rng(seed)
    T = 1 if targets is None else len(set(targets))
    pos, ang, tg = random_state(rng, E, N, T, spread)
    env = gym_macm.BatchedFlock(E, n_agents=[N], targets=targets, device="cuda:0", seed=None,
                                max_contacts=max_contacts, max_touching=max_touching, **kw)
    env.load_state(pos, ang, targets=tg)
    ref = oracle.OracleBatch(E, n_agents=N, n_targets=T, **oracle_kwargs(kw))
    ref.reset(pos, ang, targets=tg, target_idx=targets)
    return env, ref, rng


def oracle_kwargs(kw):
    """BatchedFlock settings keywords -> the OracleBatch parameters they set."""
    okw = {}
    if "reward_mode" in kw: okw["reward_mode"] = {"binary": 0, "linear": 1}[kw["reward_mode"]]
    if "action_mode" in kw: okw["action_mode"] = {"discrete": 0, "continuous": 1}[kw["action_mode"]]
    if "coord" in kw: okw["coord"] = {"polar": 0, "cartesian": 1}[kw["coord"]]
    if "damping_model" in kw: okw["damping_model"] = {"taylor": 0, "pade": 1}[kw["damping_model"]]
    for k_, ok in (("time_limit", "time_limit"), ("hz", "hz"), ("velocityIterations", "velocity_iterations"),
                   ("positionIterations", "position_iterations"), ("agent_force", "agent_force"),
                   ("_reward_radius", "reward_radius"), ("enableWarmStarting", "warm_starting")):
        if k_ in kw: okw[ok] = kw[k_]
    return okw


def run_parity(E, N, steps, targets=None, seed=0, spread=20.0, policy="random", check_every=1, **kw):
    import torch
    env, ref, rng = make_pair(E, N, targets, seed, spread, **kw)
    coord, rmode = kw.get("coord", "polar"), kw.get("reward_mode", "binary")
    cont = kw.get("action_mode", "discrete") == "continuous"
    # initial observation (Flock.__init__ -> get_obs, mvmnt.py:79)
    torch.cuda.synchronize()
    compare_obs(env.state["obs"].cpu().numpy(), ref.flock_observe(), coord)
    stats = dict(max_contacts=0, max_touching=0, multi=0)
    for k in range(steps):
        if cont:
            # the tensor API takes float32 actions; the oracle gets the same values widened
            act = rng.uniform(-1.2, 1.2, (E, N, 2)).astype(np.float32).astype(np.float64)
            env.step(torch.as_tensor(act, dtype=torch.float32, device="cuda:0"))
            o = ref.flock_step(act)
        else:
            if policy == "random":
                act = rng.integers(0, 3, (E, N, 3))
            elif policy == "flock":   # bots.flock on the device, then the same actions to the oracle
                act = env.bot_actions("flock").cpu().numpy()[..., :3].astype(np.int64)
            elif policy == "idle":
                act = np.ones((E, N, 3), np.int64)
            env.step(torch.as_tensor(act, device="cuda:0"))
            o = ref.flock_step(act)
        if (k + 1) % check_every == 0 or k == steps - 1:
            compare_step(env, ref, o, k, coord, rmode)
        es = env.state["env_state"].cpu().numpy()
        stats["max_touching"] = max(stats["max_touching"], int(es[:, 2].max()))
        stats["max_contacts"] = max(stats["max_contacts"], int(env.state["contact_count"].max()))
    env.close()
    return stats
