"""TDM (repaired semantics, SURVEY.md Appendix B): CUDA path against the CPU oracle."""
import numpy as np
import pytest

from _parity import OBS_ATOL, OBS_RTOL, ang_diff, gpu_bodies

pytestmark = pytest.mark.gpu


def steps_left(c, hz=60.0):
    k = 0
    while c > 0:
        c -= 1 / hz
        k += 1
    return k


def tdm_spawn(rng, E, teams, width=30.0, height=30.0):
    """combat.py:84-86: x = U * (team + width/2), y = U * height; headings uniform in [-pi, pi)."""
    team = np.array([t for t, n in enumerate(teams) for _ in range(n)], np.uint8)
    N = len(team)
    pos = np.stack([rng.random((E, N)) * (team[None] + width / 2), rng.random((E, N)) * height], -1)
    ang = rng.uniform(-1, 1, (E, N)) * np.pi
    return team, pos, ang


def run_tdm(E, teams, steps, seed, width=30.0, height=30.0, attack_p=0.5, check_every=1, max_touching=None):
    """max_touching=None asks for full capacity, N(N-1)/2 (more than 240 from 23 agents on: the global-memory stage
    of macm_kernels_huge.cu); 0 is the library default."""
    import torch
    import gym_macm
    from oracle import oracle
    rng = np.random.default_rng(seed)
    team, pos, ang = tdm_spawn(rng, E, teams, width, height)
    N = len(team)
    pairs = N * (N - 1) // 2
    env = gym_macm.BatchedTDM(E, n_agents=list(teams), device="cuda:0", seed=None, max_contacts=pairs,
                              max_touching=pairs if max_touching is None else max_touching)
    env.load_state(pos, ang)
    ref = oracle.OracleBatch(E, env_kind=oracle.TDM, n_agents=N, n_targets=0)
    ref.reset(pos, ang, team=team)
    deaths = 0
    for k in range(steps):
        act = np.concatenate([rng.integers(0, 3, (E, N, 3)), (rng.random((E, N, 1)) < attack_p).astype(np.int64)], -1)
        env.step(torch.as_tensor(act, device="cuda:0"))
        o = ref.tdm_step(act)
        if (k + 1) % check_every and k != steps - 1:
            continue
        alive = compare_tdm_step(env, ref, o, k)
        deaths = int((~alive).sum())
    env.close()
    return deaths


def compare_tdm_step(env, ref, o, k, contact_envs=8, envs=None):
    """Hold a BatchedTDM to the oracle after step k (o: that step's tdm_step outputs); returns the oracle's alive
    mask [E,N].  Contact lists are compared for the first `contact_envs` envs (None: all).  envs: bool [E], the envs
    held (None: all); the others, e.g. envs that ran out of contact capacity, are left out."""
    import torch
    E, N = ref.E, ref.N
    m = np.ones(E, bool) if envs is None else np.asarray(envs, bool)
    torch.cuda.synchronize()
    st = env.state
    assert not (st["env_state"][:, 1].cpu().numpy()[m] & 6).any(), "overflow"
    gb, rb = gpu_bodies(env)[m], ref.bodies()[m]
    assert np.array_equal(gb, rb), "step %d: body state differs at (held env, agent, field) %s" % (k, np.argwhere(gb != rb)[:3])
    ts = ref.tdm_state()[m]
    tg = st["tdm_state"].cpu()[torch.as_tensor(m)]
    ti = tg.view(torch.int32).numpy()
    assert np.array_equal(tg[..., 0].numpy().astype(np.float64), ts[..., 0]), "step %d: health" % k
    assert np.array_equal((ti[..., 3] & 1), ts[..., 3].astype(np.int32)), "step %d: alive" % k
    want_atk = np.vectorize(steps_left)(ts[..., 1])
    want_mov = np.vectorize(steps_left)(ts[..., 2])
    alive = ts[..., 3] > 0
    assert np.array_equal(ti[..., 1][alive], want_atk[alive]), "step %d: attack cool-down" % k
    assert np.array_equal(ti[..., 2][alive], want_mov[alive]), "step %d: movement cool-down" % k
    assert np.array_equal(st["collided"].cpu().numpy()[m], o["collided"][m]), "step %d: collision flags" % k
    assert np.array_equal(st["rewards"].cpu().numpy().astype(np.float64)[m], o["rewards"][m]), "step %d: rewards" % k
    assert np.array_equal(st["done"].cpu().numpy()[m], o["done"][m]), "step %d: done" % k
    assert np.array_equal(st["env_state"][:, 3].cpu().numpy()[m], o["winner"][m]), "step %d: winner" % k
    obs = st["obs"].cpu().numpy().reshape(E, N, N, 4)[m]
    assert np.array_equal(obs[..., 3].astype(np.int8), o["type"][m]), "step %d: ally/enemy/none flags" % k
    t = o["type"][m] >= 0
    oo = o["obs"][m]
    assert np.allclose(obs[..., 0][t], oo[..., 0][t], rtol=OBS_RTOL, atol=OBS_ATOL)
    assert ang_diff(obs[..., 1][t].astype(np.float64), oo[..., 1][t]).max(initial=0) <= 3e-6
    assert ang_diff(obs[..., 2][t].astype(np.float64), oo[..., 2][t]).max(initial=0) <= 3e-6
    for e in range(E if contact_envs is None else min(E, contact_envs)):
        if not m[e]:
            continue
        ab, fl, imp = env.contacts(e)
        rab, rfl, rimp = ref.contacts(e)
        assert np.array_equal(ab, rab) and np.array_equal(fl, rfl), "step %d env %d: contacts" % (k, e)
        assert np.array_equal(imp[rfl.astype(bool)], rimp[rfl.astype(bool)])
    return ref.tdm_state()[..., 3] > 0


def test_tdm_duel_small():
    run_tdm(64, [2, 2], 400, seed=1, width=4.0, height=3.0, check_every=5)


def test_tdm_3x15_config4_shape():
    # BASELINE config 4: 3 teams x 15 agents (N = 45), default 30 x 30 world
    run_tdm(32, [15, 15, 15], 150, seed=2, check_every=10)


def test_tdm_crowded_many_deaths():
    # a small arena: agents in melee range all the time -> health, deaths, winners, contact destruction
    d = run_tdm(48, [6, 6, 6], 700, seed=3, width=6.0, height=6.0, attack_p=0.9, check_every=20)
    assert d > 48


def test_tdm_more_than_64_agents():
    # three teams of 30: 90 agents per arena, four agents per lane
    d = run_tdm(12, [30, 30, 30], 200, seed=5, check_every=10)
    d2 = run_tdm(8, [40, 35], 300, seed=6, width=12.0, height=12.0, attack_p=0.9, check_every=25)
    assert d + d2 > 0
