"""Final observation and outcome of a reset env (macm_bind_final, macm_rollout_out.final_*, keep_final=True): every
reset -- reset_done, the one auto_reset appends to a step or rollout, a rollout's in-launch reset -- first copies the
env's rows of obs / nn_idx / tdm_state / env_state as they stand.  Held bitwise to a twin batch without auto-reset that
snapshots its own rows and then calls reset_done with the same seed; rows of envs that are not reset stay untouched."""
import ctypes as C

import pytest

from test_gpu_rollout import _same_state

pytestmark = pytest.mark.gpu

SENT = -7          # sentinel every final array starts with: marks the rows nothing wrote
AUTO_SEED = 77
OUTS = ("obs", "nn_idx", "rewards", "collided", "done")


def _names(env):
    return [n for n in ("obs", "nn_idx", "tdm_state", "env_state") if n in env.state]


def _fill(tensors):
    for t in tensors.values():
        t.fill_(SENT)


def _rows_equal(a, b, rows):
    import torch
    return torch.equal(a[rows], b[rows])


def _twin_check(A, B, step_fn, n_steps):
    """A: auto_reset + keep_final.  B: same seed, no auto-reset; after each step B snapshots its rows and resets its
    done envs with A's auto seed.  Returns the steps at which some env finished and the envs that ever finished."""
    import torch
    names = _names(A)
    _fill(A.engine.final)
    ended, ever = [], torch.zeros(A.engine.E, dtype=torch.bool, device="cuda:0")
    for k in range(n_steps):
        step_fn(k)
        snap = {n: B.state[n].clone() for n in names}
        before = {n: A.engine.final[n].clone() for n in names}
        B.reset_done(seed=AUTO_SEED)
        d = B.done
        assert torch.equal(A.done, d), k
        for n in names:
            assert _rows_equal(A.engine.final[n], snap[n], d), (k, n)          # the finished envs' terminal rows
            assert _rows_equal(A.engine.final[n], before[n], ~d), (k, n)       # the others untouched
        _same_state(A, B, "step %d" % k)
        if bool(d.any()):
            ended.append(k)
            ever |= d
    return ended, ever


@pytest.mark.parametrize("N", [64, 100, 45])     # 45: rows that are not a whole number of 16-byte vectors
@pytest.mark.parametrize("coord", ["polar", "cartesian"])
def test_single_steps_flock(N, coord):
    import torch
    import gym_macm
    E = 24
    kw = dict(n_agents=[N], device="cuda:0", seed=31, time_limit=0.2, coord=coord, start_spread=10.0)
    A = gym_macm.BatchedFlock(E, auto_reset=True, keep_final=True, **kw)
    B = gym_macm.BatchedFlock(E, **kw)
    A.engine.set_auto_reset_seed(AUTO_SEED)
    assert A.engine.info.done_step == 13
    g = torch.Generator(device="cuda:0")
    g.manual_seed(N)
    acts = torch.zeros((39, E, N, 4), dtype=torch.uint8, device="cuda:0")
    acts[..., :3] = torch.randint(0, 3, (39, E, N, 3), generator=g, device="cuda:0", dtype=torch.uint8)

    def step(k):
        A.step(acts[k])
        B.step(acts[k])
    ended, ever = _twin_check(A, B, step, 39)
    assert ended == [12, 25, 38] and bool(ever.all())      # three episodes, every env
    info = A.final_info
    assert bool((info["step_count"] == 13).all()) and bool((info["episode"] == 2).all())
    assert not bool(info["overflowed"].any())
    fo = A.final_obs
    assert fo["nodes"][0]["id"] is A.engine.final["nn_idx"] and fo["nodes"][0]["position"].shape == (E, N, 2 if coord == "polar" else 3)


def test_single_steps_tdm():
    import torch
    import gym_macm
    E = 40
    kw = dict(n_agents=[3, 3], device="cuda:0", seed=9, world_width=5.0, world_height=4.0)
    A = gym_macm.BatchedTDM(E, auto_reset=True, keep_final=True, **kw)
    B = gym_macm.BatchedTDM(E, **kw)
    A.engine.set_auto_reset_seed(AUTO_SEED)

    def step(k):
        a = A.bot_actions("combat")
        A.step(a)
        B.step(a)
    ended, ever = _twin_check(A, B, step, 400)
    assert len(ended) >= 3                                   # matches end at different steps
    info, fo = A.final_info, A.final_obs
    # a finished match has a winner unless its last agents fell together
    w = info["winner"][ever]
    assert bool(((w >= 0) == fo["alive"][ever].any(-1)).all()) and bool((w >= 0).any())
    assert torch.equal(info["episode"][ever] + 1, A.episode[ever])          # the finished episode, not the new one
    # envs whose match never ended keep the sentinel in every final array
    for n in _names(A):
        assert bool((A.engine.final[n][~ever] == SENT).all()), n


def _rollout_case(make, K, actions=None, policy=None):
    """single steps (one) vs one rollout (many) vs the same rollout with nothing bound (plain)."""
    import torch
    one, many = make(True), make(True)
    plain = make(False)
    for e in (one, many, plain):
        e.engine.set_auto_reset_seed(AUTO_SEED)
    names = _names(one)
    _fill(one.engine.final)
    _fill(many.engine.final)
    per = {n: [] for n in names}
    steps = {n: [] for n in OUTS if n in one.state}
    for k in range(K):
        a = actions[k] if actions is not None else one.bot_actions(policy, seed=5)
        one.step(a)
        for n in names:
            per[n].append(one.engine.final[n].clone())
        for n in steps:
            steps[n].append(one.state[n].clone())
    want = tuple(steps) + tuple("final_" + n for n in names)
    out = many.engine.rollout_buffers(K, want)
    _fill({n: t for n, t in out.items() if n.startswith("final_")})
    if actions is not None:
        many.rollout(actions[:K], out=out)
        ref = plain.rollout(actions[:K], want=tuple(steps))
    else:
        many.rollout(None, n_steps=K, policy=policy, seed=5, out=out)
        ref = plain.rollout(None, n_steps=K, policy=policy, seed=5, want=tuple(steps))
    torch.cuda.synchronize()
    done = out["done"].bool()
    assert bool(done.any())
    for n in names:
        got = out["final_" + n]
        for k in range(K):
            d = done[k]
            assert _rows_equal(got[k], per[n][k], d), (n, k)
            assert bool((got[k][~d] == SENT).all()), (n, k)
        assert torch.equal(one.engine.final[n], many.engine.final[n]), n      # bound slots: the latest terminal
    last = K - 1
    for n in steps:
        want_n = torch.stack(steps[n])
        if n in ("obs", "nn_idx"):
            # the launch writes its last step's observation before the reset it appends: the terminal one there
            d = done[last]
            want_n[last][d] = per[n][last][d]
        assert torch.equal(out[n], want_n), n
        assert torch.equal(out[n], ref[n]), n                                 # the terminal pass perturbs nothing
    _same_state(one, many, "rollout vs steps")
    _same_state(plain, many, "rollout vs unbound rollout")
    assert many.engine.launch_count == plain.engine.launch_count
    return done


def _flock(N=64, E=32, **kw):
    import gym_macm

    def make(keep):
        return gym_macm.BatchedFlock(E, n_agents=[N], device="cuda:0", seed=8, time_limit=0.2, auto_reset=True,
                                     keep_final=keep, start_spread=10.0, **kw)
    return make


def _acts(K, E, N, seed):
    import torch
    g = torch.Generator(device="cuda:0")
    g.manual_seed(seed)
    acts = torch.zeros((K, E, N, 4), dtype=torch.uint8, device="cuda:0")
    acts[..., :3] = torch.randint(0, 3, (K, E, N, 3), generator=g, device="cuda:0", dtype=torch.uint8)
    return acts


def test_rollout_flock_actions():
    # K = 39: the envs finish after steps 12 and 25 (in-launch resets) and 38 (the reset the launch appends)
    done = _rollout_case(_flock(), 39, actions=_acts(39, 32, 64, 1))
    assert [k for k in range(39) if bool(done[k].any())] == [12, 25, 38]


def test_rollout_flock_policy():
    _rollout_case(_flock(), 30, policy="flock")


def test_rollout_flock_huge_stage():
    # max_touching > 240 routes every step launch to the kernels with the global-memory solver stage
    make = _flock(N=64, E=16, max_touching=300)
    assert make(False).engine.sizes.touch_scratch > 0
    _rollout_case(make, 27, actions=_acts(27, 16, 64, 2))


def test_rollout_tdm_combat():
    import gym_macm

    def make(keep):
        return gym_macm.BatchedTDM(40, n_agents=[3, 3], device="cuda:0", seed=9, world_width=5.0, world_height=4.0,
                                   auto_reset=True, keep_final=keep)
    done = _rollout_case(make, 400, policy="combat")
    assert len({k for k in range(400) if bool(done[k].any())}) >= 3


def test_masked_reset_fills_only_masked_envs():
    import torch
    import gym_macm
    E, N = 16, 12
    env = gym_macm.BatchedFlock(E, n_agents=[N], device="cuda:0", seed=3, keep_final=True, start_spread=6.0)
    for k in range(5):
        env.step(_acts(1, E, N, k)[0])
    _fill(env.engine.final)
    mask = torch.zeros(E, dtype=torch.bool, device="cuda:0")
    mask[[0, 3, 4, 15]] = True
    snap = {n: env.state[n].clone() for n in _names(env)}
    env.reset_done(mask, seed=4)
    for n in _names(env):
        assert _rows_equal(env.engine.final[n], snap[n], mask), n
        assert bool((env.engine.final[n][~mask] == SENT).all()), n
    assert bool((env.final_info["step_count"][mask] == 5).all()) and bool((env.final_info["episode"][mask] == 0).all())


def test_bind_final_status_codes():
    import torch
    import gym_macm
    from gym_macm import _lib
    L = _lib.lib()
    fl = gym_macm.BatchedFlock(4, n_agents=[4], device="cuda:0", seed=0)
    td = gym_macm.BatchedTDM(4, n_agents=[2, 2], device="cuda:0", seed=0)
    buf = torch.zeros(4096, dtype=torch.float32, device="cuda:0")
    p = buf.data_ptr()

    def bind(env, **kw):
        f = _lib.MacmFinalOut(**kw)
        return L.macm_bind_final(env.engine._h, C.byref(f))
    assert bind(fl, tdm_state=p) == -1 and bind(td, nn_idx=p) == -1          # not this env kind's arrays
    assert bind(fl, obs=p + 4) == -4 and bind(fl, env_state=p + 8) == -4 and bind(td, tdm_state=p + 4) == -4
    assert bind(fl, nn_idx=p + 4) == 0 and bind(td, obs=p, tdm_state=p + 16, env_state=p + 64) == 0
    assert L.macm_bind_final(td.engine._h, None) == 0
    # rollout final arrays: the same rules
    a = torch.zeros((2, 4, 4, 4), dtype=torch.uint8, device="cuda:0")
    ro = _lib.MacmRolloutOut(final_nn_idx=p)
    assert L.macm_rollout(td.engine._h, C.c_void_p(a.data_ptr()), 2, -1, 0, C.byref(ro), None) == -1
    ro = _lib.MacmRolloutOut(final_obs=p + 4)
    assert L.macm_rollout(fl.engine._h, C.c_void_p(a.data_ptr()), 2, -1, 0, C.byref(ro), None) == -4
    with pytest.raises(_lib.MacmError):
        fl.final_obs
    # unbinding: a reset copies nothing
    fl.engine.bind_final()
    _fill(fl.engine.final)
    assert L.macm_bind_final(fl.engine._h, None) == 0
    fl.reset_done(torch.ones(4, dtype=torch.bool, device="cuda:0"))
    torch.cuda.synchronize()
    assert all(bool((t == SENT).all()) for t in fl.engine.final.values())


def test_final_nn_idx_needs_only_word_alignment():
    """nn_idx arrays (bound or final) need 4-byte alignment only: a final nn_idx 4 bytes past a 16-byte boundary is
    filled correctly by reset_done and by the reset a rollout appends (N = 64: whole 16-byte vectors per row)."""
    import torch
    import gym_macm
    from gym_macm import _lib
    E, N, K = 8, 64, 13
    env = gym_macm.BatchedFlock(E, n_agents=[N], device="cuda:0", seed=5, time_limit=0.2, auto_reset=True,
                                start_spread=10.0)
    L = _lib.lib()
    raw = torch.full((E * N + 4,), SENT, dtype=torch.int32, device="cuda:0")
    assert raw.data_ptr() % 16 == 0
    fin_nn = raw[1:1 + E * N].view(E, N)                    # 4 bytes past the boundary
    fin_es = torch.full((E, 4), SENT, dtype=torch.int32, device="cuda:0")
    f = _lib.MacmFinalOut(nn_idx=fin_nn.data_ptr(), env_state=fin_es.data_ptr())
    assert L.macm_bind_final(env.engine._h, C.byref(f)) == 0
    acts = _acts(K, E, N, 3)
    for k in range(3):
        env.step(acts[k])
    mask = torch.zeros(E, dtype=torch.bool, device="cuda:0")
    mask[[1, 6]] = True
    snap = env.state["nn_idx"].clone()
    env.reset_done(mask, seed=2)
    torch.cuda.synchronize()
    assert torch.equal(fin_nn[mask], snap[mask]) and bool((fin_nn[~mask] == SENT).all())
    assert bool((fin_es[mask][:, 0] == 3).all())
    # a rollout of K = 13 steps: the envs just reset finish on its last step (the reset the launch appends copies
    # row K-1 through the word-aligned final_nn_idx), the others after step 9 (the in-launch reset)
    raw_k = torch.full((K * E * N + 4,), SENT, dtype=torch.int32, device="cuda:0")
    out_nn = raw_k[1:1 + K * E * N].view(K, E, N)
    out = env.engine.rollout_buffers(K, ("nn_idx", "done"))
    out["final_nn_idx"] = out_nn
    env.rollout(acts, out=out)
    torch.cuda.synchronize()
    d = out["done"].bool()
    assert torch.equal(d[K - 1], mask) and torch.equal(d[9], ~mask)
    assert torch.equal(out_nn[K - 1][mask], out["nn_idx"][K - 1][mask])     # the launch's last step: terminal obs
    assert torch.equal(fin_nn[mask], out["nn_idx"][K - 1][mask])
    assert torch.equal(out_nn[9][~mask], fin_nn[~mask])                      # bound slot: the latest terminal
    for k in range(K):
        assert bool((out_nn[k][~d[k]] == SENT).all()), k


def test_launch_count_unchanged_by_binding():
    import gym_macm
    E, N = 8, 8
    envs = [gym_macm.BatchedFlock(E, n_agents=[N], device="cuda:0", seed=1, time_limit=0.05, auto_reset=True,
                                  keep_final=keep) for keep in (False, True)]
    acts = _acts(6, E, N, 0)
    for e in envs:
        for k in range(6):
            e.step(acts[k])
        e.rollout(acts)
        e.reset_done()
    assert envs[0].engine.launch_count == envs[1].engine.launch_count
