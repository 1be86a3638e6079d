"""macm_render_agents on the device against the float64 restatement of its drawing rules
(test_agent_frames_cpu.rasterize_agent): every agent's frame of stepped Flock batches at every dispatched agent count
and of TDM batches with dead agents, sizes from 1 x 1 to 1024 x 1024, env lists in any order; the call reads the state
and writes nothing else; it is ordered on the batch's stream; the ABI's errors and its black frames for bad device
data."""
import ctypes as C

import numpy as np
import pytest

from test_agent_frames_cpu import rasterize_agent

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _check(env, frames, envs, half_width, size, max_ambiguous=1e-2):
    """Frame (b, i) equals the restatement of agent i of env envs[b] on every non-ambiguous pixel.  Ambiguous pixels
    are under 1 % of the frame beside those along the observer's own heading axis: in a frame of even width that
    axis runs on a pixel boundary, exactly 0.5 px from the centres on either side of it."""
    from gym_macm import render
    got = frames.cpu().numpy()
    N = env.engine.N
    H, W = size
    assert got.shape == (len(envs), N, H, W, 3)
    rho = env.settings.bodySettings["fixtures"].radius * W / (2.0 * half_width)
    allowed = max_ambiguous * H * W + 2 * (np.ceil(rho) + 2)
    for b, e in enumerate(envs):
        fr = render.export(env, int(e))
        for i in range(N):
            ref, amb = rasterize_agent(fr, i, half_width, size)
            bad = (got[b, i] != ref).any(-1) & ~amb
            assert not bad.any(), "frame (%d, %d) (env %d): %d pixels differ, first at %s" % (
                b, i, e, bad.sum(), np.argwhere(bad)[0])
            assert amb.sum() <= allowed, "frame (%d, %d): %d ambiguous pixels" % (b, i, amb.sum())


def _flock(E, N, T, steps=30, seed=1, spread=None, **kw):
    """A Flock batch stepped by the `flock` and `random` actors in turn (contacts and a gathering flock)."""
    import torch
    import gym_macm
    spread = spread if spread is not None else max(2.5, np.sqrt(N))
    env = gym_macm.BatchedFlock(E, n_agents=[N], targets=[i % T for i in range(N)], device=DEV, seed=seed,
                                start_spread=spread, **kw)
    for k in range(steps):
        env.step(env.bot_actions("flock" if k % 2 else "random", seed=k))
    torch.cuda.synchronize()
    return env


def _tdm(E, teams, seed=3):
    import torch
    import gym_macm
    env = gym_macm.BatchedTDM(E, n_agents=teams, device=DEV, seed=seed, world_width=8, world_height=8)
    for _ in range(20):
        env.rollout(None, n_steps=100, policy="combat", seed=seed, want=())
        if int((~env.alive).sum(1).gt(0).sum()) >= E // 2:
            break
    torch.cuda.synchronize()
    return env


@pytest.mark.parametrize("N,T", [(4, 1), (6, 3), (16, 4), (32, 16), (64, 16), (64, 2), (128, 16)])
def test_flock_frames(N, T):
    E = 4
    env = _flock(E, N, T)
    assert bool(env.collided.any()), "the case should show agents in a contact"
    for size, hw in (((16, 16), 3.0), ((84, 84), 6.0), ((7, 5), 2.0)):
        frames = env.render_agents(size, hw)
        _check(env, frames, range(E), hw, size)
    envs = [2, 0, 2]
    frames = env.render_agents((32, 32), 10.0, envs=envs)
    _check(env, frames, envs, 10.0, (32, 32))


def test_tdm_frames_with_deaths():
    import torch
    E = 4
    env = _tdm(E, [5, 5, 4, 2])          # a fourth team: the grey of teams beyond combat.py's three
    assert bool((~env.alive).any()), "the case should show dead agents"
    for size, hw in (((32, 32), 4.0), ((84, 84), 8.0)):
        frames = env.render_agents(size, hw)
        _check(env, frames, range(E), hw, size)
        assert frames.cpu().numpy()[(~env.alive).cpu().numpy()].any(axis=(1, 2, 3)).all(), "dead agents keep frames"
    envs = torch.tensor([3, 1, 1], device=DEV, dtype=torch.int32)
    frames = env.render_agents((16, 16), 5.0, envs=envs)
    _check(env, frames, envs.tolist(), 5.0, (16, 16))


@pytest.mark.parametrize("size", [(1, 1), (7, 5), (16, 16), (84, 84), (1024, 1024)])
def test_sizes(size):
    env = _flock(4, 16, 2, steps=10)
    envs = [1, 3] if size == (1024, 1024) else [3, 0, 2, 0]
    frames = env.render_agents(size, 4.0, envs=envs)
    # in a 1 x 1 frame one ambiguous pixel is the whole frame: it is only left out of the comparison
    _check(env, frames, envs, 4.0, size, max_ambiguous=1.0 if size == (1, 1) else 1e-2)
    if size == (1, 1):
        # the one pixel sits on each observer's own centre, on its heading axis, unless a later primitive covers it
        assert frames.cpu().numpy().any(axis=(2, 3, 4)).all()


def test_envs_none_list_and_tensor_agree():
    import torch
    env = _flock(5, 32, 3, steps=12)
    every = env.render_agents((32, 32), 5.0)
    listed = env.render_agents((32, 32), 5.0, envs=[4, 4, 0, 2])
    tensor = env.render_agents((32, 32), 5.0, envs=torch.tensor([4, 4, 0, 2], device=DEV))
    assert torch.equal(listed, every[[4, 4, 0, 2]]) and torch.equal(tensor, listed)
    assert torch.equal(env.render_agents((32, 32), 5.0, envs=range(5)), every)


def test_render_agents_is_read_only():
    import torch
    a, b = _flock(8, 16, 2, steps=12, seed=5), _flock(8, 16, 2, steps=12, seed=5)
    before = {n: t.clone() for n, t in a.engine.t.items()}
    launches = a.engine.launch_count
    out = torch.full((8, 16, 32, 32, 3), 7, dtype=torch.uint8, device=DEV)
    assert a.render_agents((32, 32), 5.0, out=out) is out
    torch.cuda.synchronize()
    assert a.engine.launch_count == launches + 1
    for n, t in a.engine.t.items():
        assert torch.equal(t, before[n]), n
    acts = torch.randint(0, 3, (8, 16, 3), device=DEV)
    a.step(acts)
    b.step(acts)
    torch.cuda.synchronize()
    for n in a.engine.t:
        assert torch.equal(a.engine.t[n], b.engine.t[n]), n


def test_stream_order():
    import torch
    import gym_macm
    E, N, size, hw = 8, 16, (16, 16), 4.0
    s = torch.cuda.Stream(device=DEV)
    env = gym_macm.BatchedFlock(E, n_agents=[N], device=DEV, seed=9, start_spread=5.0, stream=s)
    acts = [torch.randint(0, 3, (E, N, 3), device=DEV) for _ in range(6)]
    s.wait_stream(torch.cuda.current_stream(DEV))
    for a in acts:
        env.step(a)
    frames = env.render_agents(size, hw)      # right after the step, on the batch's stream, no sync in between
    s.synchronize()
    _check(env, frames, range(E), hw, size)

    pool = gym_macm.BatchPool([gym_macm.BatchedFlock(E, n_agents=[N], device=DEV, seed=20 + r, start_spread=5.0)
                               for r in range(2)])
    packed = [pool.batches[0].pack_actions(a).clone() for a in acts]
    torch.cuda.synchronize()
    last = {}
    for k, a in enumerate(packed):
        b = pool.step(a)
        last[k % 2] = (b, b.render_agents(size, hw))
    pool.synchronize()
    for b, frames in last.values():
        _check(b, frames, range(E), hw, size)


def test_errors_and_black_frames():
    import torch
    from gym_macm import _lib, render
    L = _lib.lib()
    env = _flock(4, 8, 1, steps=3)
    E, N, h = 4, 8, env.engine._h
    pal = torch.from_numpy(render.palette(env)).to(DEV)
    out = torch.zeros((6, N, 16, 16, 3), dtype=torch.uint8, device=DEV)
    stream = C.c_void_p(torch.cuda.current_stream(DEV).cuda_stream)

    def call(n=4, H=16, W=16, hw=3.0, envs=None, p=pal, o=out, handle=h, envs_ptr=None):
        ep = envs_ptr if envs_ptr is not None else (None if envs is None else envs.data_ptr())
        a = _lib.MacmAgentFramesArgs(n, H, W, hw, ep, None if p is None else p.data_ptr(),
                                     None if o is None else o.data_ptr())
        return L.macm_render_agents(handle, C.byref(a), stream)

    assert call() == 0
    for bad in (dict(n=0), dict(n=5), dict(H=0), dict(W=0), dict(W=1025), dict(H=1025), dict(hw=0.0), dict(hw=-1.0),
                dict(hw=float("inf")), dict(hw=float("nan")), dict(p=None), dict(o=None)):
        assert call(**bad) == -1, bad                           # MACM_E_INVALID
    idx = torch.zeros(8, dtype=torch.int32, device=DEV)
    assert call(n=2, envs_ptr=idx.data_ptr() + 2) == -4         # MACM_E_ALIGN
    p = _lib.default_params(_lib.FLOCK)
    unbound = C.c_void_p()
    assert L.macm_create(C.byref(unbound), C.byref(p), 0) == 0
    try:
        assert call(handle=unbound) == -3                       # MACM_E_UNBOUND
    finally:
        L.macm_destroy(unbound)
    # from Python: bad indices, sizes, half-widths and outputs raise before the call
    for kw in (dict(envs=[0, E]), dict(envs=[-1]), dict(envs=torch.tensor([1, 9], device=DEV))):
        with pytest.raises(ValueError):
            env.render_agents((16, 16), 3.0, **kw)
    for size, hw in (((0, 16), 3.0), ((16, 1025), 3.0), ((16, 16), 0.0), ((16, 16), float("nan"))):
        with pytest.raises(ValueError):
            env.render_agents(size, hw)
    for o in (torch.zeros((4, N, 16, 16, 3), dtype=torch.uint8), torch.zeros((4, N, 16, 16, 3), device=DEV),
              torch.zeros((4, N, 16, 17, 3), dtype=torch.uint8, device=DEV)):
        with pytest.raises(ValueError):
            env.render_agents((16, 16), 3.0, out=o)
    # the same indices straight to the ABI: N black frames per bad row, nothing read out of bounds
    envs = torch.tensor([-1, E, 1 << 30, -(1 << 31), 0, 2], dtype=torch.int32, device=DEV)
    out.fill_(9)
    assert call(n=6, envs=envs) == 0
    torch.cuda.synchronize()
    o = out.cpu().numpy()
    assert not o[:4].any()
    _check(env, out[4:], [0, 2], 3.0, (16, 16))
