"""16-bit observations (`obs_dtype="float16" | "bfloat16"`) against an fp32 twin.

A twin batch is built from the same spawn and stepped with the same actions, one at obs_dtype float32 (held to the
oracle by the rest of the suite) and one at a 16-bit type.  On every step, every state buffer and rewards / nn_idx /
collided / done / env_state must be bit-identical between the twins, and every 16-bit observation must be exactly the
fp32 one rounded to nearest even: obs16.view(int16) == obs32.to(dtype).view(int16).  The same holds for every other
place an observation is written: rollout per-step rows, final rows, observe, resets, the host path and peer stores.
"""
import ctypes as C
import functools
import os
import socket

import numpy as np
import pytest
import torch

from test_gpu_kernel_matrix import CASES, _case_id, _launch, _make, block_threads  # noqa: F401 (fixture)

pytestmark = pytest.mark.gpu

DTYPES = ("float16", "bfloat16")
DEV = "cuda:0"


def _rounded(o32, o16, dtype, what):
    want = o32.to(getattr(torch, dtype))
    assert o16.dtype == want.dtype, what
    assert torch.equal(o16.view(torch.int16), want.view(torch.int16)), what


def _twins(s32, s16, dtype, what):
    """Every bound buffer of the twins: bit-identical, obs rounded."""
    for n, t in s32.engine.t.items():
        if n == "touch_scratch":
            continue
        if n == "obs":
            _rounded(t, s16.engine.t[n], dtype, "%s: obs" % what)
        else:
            assert torch.equal(t, s16.engine.t[n]), "%s: %s" % (what, n)


def _outs(o32, o16, dtype, what):
    for n, t in o32.items():
        if n.endswith("obs"):
            _rounded(t, o16[n], dtype, "%s: %s" % (what, n))
        else:
            assert torch.equal(t, o16[n]), "%s: %s" % (what, n)


def _zero_buffers(eng, K, want):
    return {n: torch.zeros_like(t) for n, t in eng.rollout_buffers(K, want).items()}


# ---- every dispatched kernel: single steps, one-step rollouts (per-step stores), multi-step rollouts ---------------
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("c", CASES, ids=[_case_id(c) for c in CASES])
def test_kernel_twins(c, dtype, block_threads, monkeypatch):  # noqa: F811
    import gym_macm
    threads, E, mt = _launch(c)
    block_threads(threads)
    N = c["N"]
    seed = 1000 * c["G"] + 10 * c["APL"] + N + (7 if c["kind"] == "tdm" else 0)
    (one, roll, step1), _, kw = _make(c, E, mt, np.random.default_rng(seed))
    cls = "BatchedFlock" if c["kind"] == "flock" else "BatchedTDM"
    monkeypatch.setattr(gym_macm, cls, functools.partial(getattr(gym_macm, cls), obs_dtype=dtype))
    (one16, roll16, step16), _, _ = _make(c, E, mt, np.random.default_rng(seed))
    monkeypatch.undo()
    assert one16.engine.t["obs"].dtype == getattr(torch, dtype)
    assert 2 * one16.engine.sizes.obs == one.engine.sizes.obs and one16.engine.obs_dim == one.engine.obs_dim
    _twins(one, one16, dtype, "load_state")
    rng = np.random.default_rng(seed + 1)
    cont = kw.get("action_mode") == "continuous"
    chunk = []
    for k in range(32):
        if cont:
            a = torch.as_tensor(rng.uniform(-1.2, 1.2, (E, N, 2)).astype(np.float32), device=DEV)
        else:
            a = rng.integers(0, 3, (E, N, 4))
            a[..., 3] = 0 if c["kind"] == "flock" else rng.random((E, N)) < 0.6
            a = torch.as_tensor(a.astype(np.uint8), device=DEV)
        one.step(a)
        one16.step(a)
        _twins(one, one16, dtype, "step %d" % k)
        o1, o16 = step1.rollout(a[None]), step16.rollout(a[None])     # MODE 2: the per-step stores
        _outs(o1, o16, dtype, "one-step rollout %d" % k)
        _twins(step1, step16, dtype, "one-step rollout %d" % k)
        chunk.append(a)
        if len(chunk) == 16:
            acts = torch.stack(chunk)
            r1, r16 = roll.rollout(acts), roll16.rollout(acts)
            _outs(r1, r16, dtype, "rollout up to step %d" % k)
            _twins(roll, roll16, dtype, "rollout up to step %d" % k)
            chunk = []
    # action repeat: no per-step observation arrays, the pass runs after the last step only
    acts = torch.stack([a] * 8)
    r1, r16 = roll.rollout(acts, want=("rewards", "done")), roll16.rollout(acts, want=("rewards", "done"))
    _outs(r1, r16, dtype, "rollout without obs")
    _twins(roll, roll16, dtype, "rollout without obs")
    for s in (one, roll, step1, one16, roll16, step16):
        s.close()


# ---- TDM team shapes, 45 and 128 agents --------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("teams", [[15, 15, 15], [64, 64]], ids=["3x15", "2x64"])
def test_tdm_teams(teams, dtype):
    import gym_macm
    E = 40
    s32 = gym_macm.BatchedTDM(E, n_agents=teams, device=DEV, seed=11, world_width=12, world_height=12)
    s16 = gym_macm.BatchedTDM(E, n_agents=teams, device=DEV, seed=11, world_width=12, world_height=12, obs_dtype=dtype)
    _twins(s32, s16, dtype, "sample_reset")
    g = torch.Generator(device=DEV)
    g.manual_seed(3)
    for k in range(24):
        a = torch.randint(0, 3, (E, sum(teams), 4), generator=g, device=DEV, dtype=torch.uint8)
        a[..., 3] = torch.randint(0, 2, (E, sum(teams)), generator=g, device=DEV, dtype=torch.uint8)
        s32.step(a)
        s16.step(a)
        _twins(s32, s16, dtype, "step %d" % k)
    assert s16.obs["agents"]["position"].dtype == getattr(torch, dtype)
    s32.close()
    s16.close()


# ---- resets, final rows, observe, load_state ---------------------------------------------------------------------
def _pair(kind, dtype, E, N, **kw):
    import gym_macm
    if kind == "tdm":
        mk = lambda **x: gym_macm.BatchedTDM(E, n_agents=[N - N // 2, N // 2], device=DEV, seed=5, **kw, **x)
    else:
        mk = lambda **x: gym_macm.BatchedFlock(E, n_agents=[N], device=DEV, seed=5, start_spread=6.0, **kw, **x)
    return mk(), mk(obs_dtype=dtype)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("kind", ["polar", "cartesian", "tdm"])
def test_auto_reset_keep_final(kind, dtype):
    E, N = 24, 9      # odd N: cartesian records of 12 bytes, rows of 108 bytes
    kw = dict(auto_reset=True, keep_final=True, time_limit=0.2)
    if kind != "tdm":
        kw["coord"] = kind
    s32, s16 = _pair("tdm" if kind == "tdm" else "flock", dtype, E, N, **kw)
    s32.engine.set_auto_reset_seed(9)
    s16.engine.set_auto_reset_seed(9)
    g = torch.Generator(device=DEV)
    g.manual_seed(1)
    resets = 0
    for k in range(30):
        a = torch.randint(0, 3, (E, N, 4), generator=g, device=DEV, dtype=torch.uint8)
        s32.step(a)
        s16.step(a)
        resets += int(s32.done.sum())
        _twins(s32, s16, dtype, "step %d" % k)
        _outs(s32.engine.final, s16.engine.final, dtype, "final after step %d" % k)
    assert resets > 0
    # a rollout with per-step rows, final rows (in-launch resets and the appended one) and the bound final slots
    # every env is at the same step of its episode: a reset inside the launch and one after its last step
    d, c = s32.engine.info.done_step, int(s32.step_count.max())
    assert int(s32.step_count.min()) == c
    K = (d - c) + d
    acts = torch.randint(0, 3, (K, E, N, 4), generator=g, device=DEV, dtype=torch.uint8)
    want = ("obs", "nn_idx", "rewards", "collided", "done", "final_obs", "final_nn_idx", "final_tdm_state",
            "final_env_state")
    o32, o16 = _zero_buffers(s32.engine, K, want), _zero_buffers(s16.engine, K, want)
    s32.rollout(acts, out=o32)
    s16.rollout(acts, out=o16)
    assert int(o32["done"][:-1].sum()) > 0 and int(o32["done"][-1].sum()) > 0
    _outs(o32, o16, dtype, "rollout")
    _twins(s32, s16, dtype, "rollout")
    _outs(s32.engine.final, s16.engine.final, dtype, "final after rollout")
    # reset_done with a mask, observe, load_state
    mask = torch.arange(E, device=DEV) % 3 == 1
    s32.reset_done(mask, seed=4)
    s16.reset_done(mask, seed=4)
    _twins(s32, s16, dtype, "reset_done")
    _outs(s32.engine.final, s16.engine.final, dtype, "final after reset_done")
    s32.engine.t["obs"].zero_()
    s16.engine.t["obs"].zero_()
    s32.engine.observe()
    s16.engine.observe()
    _twins(s32, s16, dtype, "observe")
    rng = np.random.default_rng(2)
    pos, ang = rng.uniform(-4, 4, (E, N, 2)), rng.uniform(-np.pi, np.pi, (E, N))
    if kind == "tdm":
        s32.load_state(pos, ang)
        s16.load_state(pos, ang)
    else:
        tg = rng.uniform(-30, 30, (E, 1, 2))
        s32.load_state(pos, ang, targets=tg)
        s16.load_state(pos, ang, targets=tg)
    _twins(s32, s16, dtype, "load_state")
    # a small angle: fp16 subnormals round as torch rounds them
    if kind != "tdm":
        pos[0, 0], pos[0, 1], ang[0, 0] = (0.0, 0.0), (50.0, 1e-6), 0.0
        s32.load_state(pos, ang, targets=tg)
        s16.load_state(pos, ang, targets=tg)
        _twins(s32, s16, dtype, "load_state, small angle")
    s32.close()
    s16.close()


# ---- the host-buffer path ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("kind", ["polar", "cartesian", "tdm"])
def test_step_host(kind, dtype):
    E, N = 64, 7
    kw = {} if kind == "tdm" else {"coord": kind}
    s32, s16 = _pair("tdm" if kind == "tdm" else "flock", dtype, E, N, **kw)
    # the outputs lie back to back in one device slab and one pinned slab: one device->host copy per step
    lay = s16.engine._out_layout
    assert lay["obs"] == (0, E * N * s16.engine.obs_dim * 2)
    g = torch.Generator()
    g.manual_seed(8)
    want = ("obs", "rewards", "nn_idx", "collided", "done")
    for k in range(6):
        a = torch.randint(0, 3, (E, N, 4), generator=g, dtype=torch.uint8).pin_memory()
        wait = k % 2 == 0
        p32 = s32.engine.step_host(a, want=want, wait=wait)
        if not wait:
            s32.engine.host_sync()
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            p16 = s16.engine.step_host(a, want=want, wait=wait)
            if not wait:
                s16.engine.host_sync()
            torch.cuda.synchronize()
        d2h = [e for e in prof.events() if "DtoH" in e.name or "Device -> Pinned" in e.name]
        assert len(d2h) == 1, [e.name for e in prof.events() if "emcpy" in e.name]
        for n in want:
            if n in p32:
                if n == "obs":
                    _rounded(p32[n], p16[n], dtype, "step_host %d" % k)
                else:
                    assert torch.equal(p32[n], p16[n]), (k, n)
        _twins(s32, s16, dtype, "step_host %d" % k)
        _rounded(s32.engine.t["obs"].cpu(), p16["obs"], dtype, "pinned obs %d" % k)
    s32.close()
    s16.close()


# ---- alignment of the 16-bit records -----------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("kind", ["polar", "cartesian", "tdm"])
def test_alignment(kind, dtype):
    from gym_macm import _lib
    E, N = 8, 5
    kw = {} if kind == "tdm" else {"coord": kind}
    s32, s16 = _pair("tdm" if kind == "tdm" else "flock", dtype, E, N, **kw)
    L = _lib.lib()
    align = 4 if kind == "cartesian" else 8
    for s, a in ((s16, align), (s32, 16)):
        eng = s.engine
        raw = torch.zeros(eng.sizes.obs + 128, dtype=torch.uint8, device=DEV)
        base = (raw.data_ptr() + 63) // 64 * 64
        bufs = _lib.MacmBuffers()
        for n in _lib.BUFFER_NAMES:
            if n in eng.t:
                setattr(bufs, n, eng.t[n].data_ptr())
        fin = _lib.MacmFinalOut()
        ro = _lib.MacmRolloutOut()
        for off, want in ((a, 0), (a + 2, -4), (8, 0 if a <= 8 else -4)):
            bufs.obs = base + off
            assert L.macm_bind(eng._h, C.byref(bufs)) == want, (kind, dtype, a, off)
            fin.obs = base + off
            assert L.macm_bind_final(eng._h, C.byref(fin)) == want, (kind, dtype, a, off)
            ro.obs = base + off
            if want:   # (an aligned one would launch: covered by the rollout tests)
                rc = L.macm_rollout(eng._h, None, 1, _lib.BOTS["idle"], 0, C.byref(ro), None)
                assert rc == -4, (kind, dtype, off, rc)
            ro.obs = None
            ro.final_obs = base + off
            if want:
                rc = L.macm_rollout(eng._h, None, 1, _lib.BOTS["idle"], 0, C.byref(ro), None)
                assert rc == -4, (kind, dtype, off, rc)
            ro.final_obs = None
        bufs.obs = eng.t["obs"].data_ptr()
        _lib.check(L.macm_bind(eng._h, C.byref(bufs)))
        _lib.check(L.macm_bind_final(eng._h, None))
    s32.close()
    s16.close()


# ---- scripted actors ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", DTYPES)
def test_actors(dtype):
    from gym_macm import _lib
    E, N = 32, 6
    f32, f16 = _pair("flock", dtype, E, N)
    t32, t16 = _pair("tdm", dtype, E, N, world_width=6.0, world_height=6.0)
    # the actors that decide from the stored observation refuse a rounded one
    with pytest.raises(_lib.MacmError, match=r"status -6"):
        f16.bot_actions("flock")
    with pytest.raises(_lib.MacmError, match=r"status -6"):
        t16.bot_actions("combat")
    with pytest.raises(_lib.MacmError, match=r"status -6"):
        f16.rollout(None, 4, policy="flock")
    # the others give the fp32 twin's actions and trajectory
    for policy in ("idle", "forward", "rotate", "diag", "random", "circle"):
        assert torch.equal(f32.bot_actions(policy, seed=3), f16.bot_actions(policy, seed=3)), policy
        assert torch.equal(t32.bot_actions(policy, seed=3), t16.bot_actions(policy, seed=3)), policy
    o32, o16 = f32.rollout(None, 12, policy="random", seed=2), f16.rollout(None, 12, policy="random", seed=2)
    _outs(o32, o16, dtype, "random rollout")
    _twins(f32, f16, dtype, "random rollout")
    o32, o16 = t32.rollout(None, 80, policy="combat", seed=2), t16.rollout(None, 80, policy="combat", seed=2)
    assert bool((t32.health < 1).any()), "no strike landed"
    _outs(o32, o16, dtype, "combat rollout")
    _twins(t32, t16, dtype, "combat rollout")
    for s in (f32, f16, t32, t16):
        s.close()


# ---- PeerGather: peer stores of 16-bit observations --------------------------------------------------------------
def _worker(rank, world, port, q):
    try:
        import torch.distributed as dist
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
        dist.init_process_group("gloo", rank=rank, world_size=world)
        import gym_macm
        from gym_macm.dist import PeerGather, shard_range
        total, N = 24, 16
        start, count = shard_range(total, rank, world)
        torch.cuda.set_device(0)
        ok = []
        for dtype in DTYPES:
            env = gym_macm.BatchedFlock(count, n_agents=[N], device=DEV, seed=3, env_index_base=start, start_spread=6.0,
                                        obs_dtype=dtype)
            twin = gym_macm.BatchedFlock(count, n_agents=[N], device=DEV, seed=3, env_index_base=start,
                                         start_spread=6.0)
            pg = PeerGather(env, total, learner=0, names=("obs", "nn_idx", "rewards", "collided", "done"))
            g = torch.Generator(device=DEV)
            g.manual_seed(5)
            good = pg.full[0]["obs"].dtype == getattr(torch, dtype)
            for k in range(8):
                a_all = torch.zeros((total, N, 4), dtype=torch.uint8, device=DEV)
                a_all[..., :3] = torch.randint(0, 3, (total, N, 3), generator=g, device=DEV, dtype=torch.uint8)
                a = a_all[start:start + count].contiguous()
                pg.step(a)
                twin.step(a)
                pg.fence()
                good = good and torch.equal(env.state["obs"].view(torch.int16),
                                            twin.state["obs"].to(getattr(torch, dtype)).view(torch.int16))
                for n in pg.names:
                    mine = env.state[n].cpu()
                    if n == "obs":   # gathered as raw bytes: gloo has no 16-bit integer type
                        mine = mine.view(torch.uint8)
                    parts = [torch.empty((shard_range(total, r, world)[1],) + tuple(mine.shape[1:]), dtype=mine.dtype)
                             for r in range(world)]
                    dist.all_gather(parts, mine)
                    if rank == 0:
                        got = pg.gathered()[n].cpu()
                        good = good and torch.equal(got.view(torch.uint8) if n == "obs" else got, torch.cat(parts))
                dist.barrier()
            pg.close()
            env.close()
            twin.close()
            ok.append(bool(good))
        q.put((rank, ok))
        dist.barrier()
        dist.destroy_process_group()
    except Exception as ex:   # report instead of hanging the parent
        q.put((rank, repr(ex)))


def test_peer_gather_16_bit():
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=240) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    assert res == [(0, [True, True]), (1, [True, True])], res
