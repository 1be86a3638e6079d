"""macm_render on the device against the float64 restatement of its drawing rules (test_raster_cpu.rasterize): frames
of stepped Flock and TDM batches, every size from 1 x 1 to 2048 x 2048, fitted and cut views, env lists in any order;
render reads the state and writes nothing else; it is ordered on the batch's stream; the drop-in envs' rgb_array; the
ABI's errors and its black frames for bad device data."""
import ctypes as C

import numpy as np
import pytest

from test_raster_cpu import rasterize

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _check(env, frames, envs, views, size, max_ambiguous=1e-3):
    """Every frame equals the restatement on every non-ambiguous pixel; ambiguous pixels are under 0.1 %."""
    from gym_macm import render
    got = frames.cpu().numpy()
    views = np.asarray(views.cpu().numpy() if hasattr(views, "cpu") else views, np.float32)
    assert got.shape == (len(envs),) + tuple(size) + (3,)
    for b, e in enumerate(envs):
        ref, amb = rasterize(render.export(env, int(e)), views[b], size)
        bad = (got[b] != ref).any(-1) & ~amb
        assert not bad.any(), "frame %d (env %d): %d pixels differ, first at %s" % (b, e, bad.sum(), np.argwhere(bad)[0])
        assert amb.sum() <= max_ambiguous * amb.size, "frame %d: %d ambiguous pixels" % (b, amb.sum())


def _flock(E, N, T, coord="polar", mode="binary", steps=30, seed=1, spread=None, **kw):
    import torch
    import gym_macm
    spread = spread if spread is not None else max(4.0, 1.2 * np.sqrt(N))
    env = gym_macm.BatchedFlock(E, n_agents=[N], targets=[i % T for i in range(N)], device=DEV, seed=seed, coord=coord,
                                reward_mode=mode, start_spread=spread, **kw)
    g = torch.Generator(device=DEV).manual_seed(seed)
    for k in range(steps):
        if coord == "polar" and k % 2:
            a = env.bot_actions("flock", seed=k)
        else:
            a = torch.randint(0, 3, (E, N, 3), device=DEV, generator=g)
        env.step(a)
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


@pytest.mark.parametrize("N,T,coord,mode", [(4, 1, "polar", "binary"), (16, 4, "cartesian", "linear"),
                                            (64, 16, "polar", "linear"), (64, 2, "cartesian", "binary"),
                                            (128, 16, "polar", "binary"), (128, 3, "cartesian", "linear")])
def test_flock_frames(N, T, coord, mode):
    from gym_macm import render
    E = 6
    env = _flock(E, N, T, coord, mode)
    assert bool(env.collided.any()), "the case should show collided agents"
    for size in ((84, 84), (64, 96)):
        frames = env.render(size)
        _check(env, frames, range(E), render.fit_views(env, None, size), size)
    envs = [4, 0, 4, 5, 1, 1]
    frames = env.render((480, 640), envs=envs)
    _check(env, frames, envs, render.fit_views(env, envs, (480, 640)), (480, 640))


def test_tdm_frames_with_deaths():
    import torch
    from gym_macm import render
    E = 6
    env = _tdm(E, [5, 5, 4, 2])          # a fourth team: the grey of teams beyond combat.py's three
    assert bool((~env.alive).any()), "the case should show dead agents"
    for size in ((84, 84), (480, 640)):
        frames = env.render(size)
        _check(env, frames, range(E), render.fit_views(env, None, size), size)
    envs = torch.tensor([5, 2, 2, 0], device=DEV, dtype=torch.int32)
    frames = env.render((64, 96), envs=envs)
    _check(env, frames, envs.tolist(), render.fit_views(env, envs, (64, 96)), (64, 96))


@pytest.mark.parametrize("size", [(1, 1), (64, 96), (3, 7), (480, 640), (2048, 2048)])
def test_sizes(size):
    from gym_macm import render
    env = _flock(4, 16, 2, steps=10)
    envs = [2] if size == (2048, 2048) else [3, 0, 2]
    frames = env.render(size, envs=envs)
    # a fitted 1 x 1 frame shrinks every primitive below 1e-3 px^2: its one pixel is ambiguous, and only compared
    _check(env, frames, envs, render.fit_views(env, envs, size), size, max_ambiguous=1.0 if size == (1, 1) else 1e-3)
    if size == (1, 1):   # views centred on agent 3 of each env, then 0.2 m off it: the pixel shows its disc
        pv = env.state["posvel"][envs, 3, 0:2].cpu().numpy()
        for off in (0.0, 0.2):
            views = np.stack([pv[:, 0] + off, pv[:, 1], np.full(len(envs), 0.1)], 1).astype(np.float32)
            frames = env.render(size, envs=envs, views=views)
            _check(env, frames, envs, views, size)
            assert frames.cpu().numpy().any(axis=(1, 2, 3)).all()


def test_views_cut_agents_at_the_border():
    env = _flock(3, 16, 2, steps=10, spread=6.0)
    pv = env.state["posvel"].cpu().numpy()
    for size in ((84, 84), (60, 100)):
        # each frame's left / top / right edge runs through an agent's centre (half-height = half-width * H / W)
        hh = 3.0 * size[0] / size[1]
        views = np.array([[pv[0, 0, 0] + 2.0, pv[0, 0, 1], 2.0],
                          [pv[1, 3, 0], pv[1, 3, 1] - hh, 3.0],
                          [pv[2, 5, 0] - 1.0, pv[2, 5, 1] + 0.3, 1.0]], np.float32)
        frames = env.render(size, views=views)
        _check(env, frames, [0, 1, 2], views, size)
        assert frames.cpu().numpy().any(axis=(1, 2, 3)).all()


def test_render_is_read_only():
    import torch
    a, b = _flock(8, 16, 2, steps=12, seed=5), _flock(8, 16, 2, steps=12, seed=5)
    before = {n: t.clone() for n, t in a.engine.t.items()}
    launches = a.engine.launch_count
    out = torch.full((8, 84, 84, 3), 7, dtype=torch.uint8, device=DEV)
    assert a.render((84, 84), out=out) is out
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
    from gym_macm import render
    E, N, size = 8, 16, (84, 84)
    s = torch.cuda.Stream(device=DEV)
    env = gym_macm.BatchedFlock(E, n_agents=[N], device=DEV, seed=9, start_spread=5.0, stream=s)
    acts = [torch.randint(0, 3, (E, N, 3), device=DEV) for _ in range(6)]
    s.wait_stream(torch.cuda.current_stream(DEV))
    for a in acts:
        env.step(a)
    frames = env.render(size)                 # right after the step, on the batch's stream, no sync in between
    s.synchronize()
    _check(env, frames, range(E), render.fit_views(env, None, size), size)

    pool = gym_macm.BatchPool([gym_macm.BatchedFlock(E, n_agents=[N], device=DEV, seed=20 + r, start_spread=5.0)
                               for r in range(2)])
    packed = [pool.batches[0].pack_actions(a).clone() for a in acts]
    torch.cuda.synchronize()
    last = {}
    for k, a in enumerate(packed):
        b = pool.step(a)
        last[k % 2] = (b, b.render(size))
    pool.synchronize()
    for b, frames in last.values():
        _check(b, frames, range(E), render.fit_views(b, None, size), size)


def test_drop_in_rgb_array():
    import gym_macm
    from gym_macm.envs.combat import TDM
    from gym_macm.envs.mvmnt import Flock
    f = Flock(n_agents=[6], device=DEV, colors=[(0.1, 0.9, 0.3)] * 6)
    for _ in range(5):
        f.step({i: [1, 2, 0] for i in range(6)})
    img = f.render()
    assert img.dtype == np.uint8 and img.shape == (480, 640, 3) and img.any()
    assert np.array_equal(img, f._batch.render((480, 640))[0].cpu().numpy())
    v = (0.0, 0.0, 15.0)
    assert np.array_equal(f.render(size=(84, 84), view=v), f._batch.render((84, 84), views=[v])[0].cpu().numpy())
    with pytest.raises(NotImplementedError):
        f.render(mode="human")
    t = TDM(n_agents=[3, 3], device=DEV)
    t.step({a.id: [1, 1, 0, 1] for a in t.agents})
    assert np.array_equal(t.render(size=(120, 160)), t._batch.render((120, 160))[0].cpu().numpy())
    with pytest.raises(NotImplementedError):
        t.render(mode="human")
    assert isinstance(gym_macm.make("gym_macm:cm-flock-v0", n_agents=[3]).render(size=(8, 8)), np.ndarray)


def test_errors_and_black_frames():
    import torch
    from gym_macm import _lib, render
    L = _lib.lib()
    env = _flock(4, 8, 1, steps=3)
    E, h = 4, env.engine._h
    pal = torch.from_numpy(render.palette(env)).to(DEV)
    views = torch.tensor([[0.0, 0.0, 10.0]] * 6, device=DEV)
    out = torch.zeros((6, 16, 16, 3), dtype=torch.uint8, device=DEV)
    stream = C.c_void_p(torch.cuda.current_stream(DEV).cuda_stream)

    def call(n=4, H=16, W=16, envs=None, v=views, p=pal, o=out, handle=h):
        a = _lib.MacmRenderArgs(n, H, W, None if envs is None else envs.data_ptr(), None if v is None else v.data_ptr(),
                                None if p is None else p.data_ptr(), None if o is None else o.data_ptr())
        return L.macm_render(handle, C.byref(a), stream)

    assert call() == 0
    for bad in (dict(n=0), dict(n=5), dict(H=0), dict(W=4097), dict(H=4097), dict(v=None), dict(p=None), dict(o=None)):
        assert call(**bad) == -1, bad                           # MACM_E_INVALID
    p = _lib.default_params(_lib.FLOCK)
    unbound = C.c_void_p()
    assert L.macm_create(C.byref(unbound), C.byref(p), 0) == 0
    try:
        assert call(handle=unbound) == -3                       # MACM_E_UNBOUND
    finally:
        L.macm_destroy(unbound)
    # from Python: bad indices and views raise before the call
    for kw in (dict(envs=[0, E]), dict(envs=[-1]), dict(envs=torch.tensor([1, 9], device=DEV)),
               dict(envs=[0], views=[[0.0, 0.0, 0.0]]), dict(envs=[0], views=[[0.0, 0.0, -2.0]]),
               dict(envs=[0], views=torch.tensor([[0.0, 0.0, float("nan")]], device=DEV)),
               dict(envs=[0, 1], views=[[0.0, 0.0, 1.0]])):
        with pytest.raises(ValueError):
            env.render((16, 16), **kw)
    with pytest.raises(ValueError):
        env.render((0, 16))
    with pytest.raises(ValueError):
        env.render((16, 16), out=torch.zeros((4, 16, 16, 3), dtype=torch.uint8))
    # the same values straight to the ABI: black frames, nothing read out of bounds
    envs = torch.tensor([-1, E, 1 << 30, 0, 0, 2], dtype=torch.int32, device=DEV)
    views = torch.tensor([[0.0, 0.0, 10.0]] * 3 + [[0.0, 0.0, 0.0], [0.0, 0.0, float("inf")], [0.0, 0.0, 10.0]],
                         device=DEV)
    out.fill_(9)
    assert call(n=6, envs=envs, v=views) == 0
    torch.cuda.synchronize()
    o = out.cpu().numpy()
    assert not o[:5].any()
    _check(env, out[5:], [2], views[5:], (16, 16))
