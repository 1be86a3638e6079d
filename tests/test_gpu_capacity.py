"""Contact capacity against the oracle: max_contacts (C) and max_touching (TC, and TCH, the global-memory stage of
macm_kernels_huge.cu behind it).

The library may leave the reference in one place only: an env whose live contacts exceed C, or whose touching
contacts at Collide exceed the solver's stage, gets MACM_ENV_CONTACT_OVERFLOW / MACM_ENV_TOUCH_OVERFLOW from that step
on, and no other env is affected.  Each case below steps a pool of spawns of mixed density in the oracle first, picks
from the oracle's per-step counts a capacity that one env reaches exactly and another one exceeds, and then steps a
batch of those envs on the device:
  * the flag bits of every env that was unflagged before the step equal "the oracle's count exceeded the capacity at
    some step so far", bit by bit; set bits stay set;
  * every env that is still unflagged -- the envs that share a warp or a block with a flagged one included -- is held
    to the oracle with the usual bars; a flagged env still lists at most C pairs, each with a < b < N;
  * a multi-step rollout twin equals the single steps for every env, flagged ones included.
The last tests run the device's scripted actors at the default capacities for a whole episode: a flock that gathers
at its target packs more touching contacts than a random-action spawn ever does.
"""
import ctypes as C

import numpy as np
import pytest

from _parity import compare_step, oracle_kwargs, overflow_bits
from test_gpu_kernel_matrix import FLOCK_A, PILE, RAGGED_N, SHAPES, _launch, _teams, block_threads  # noqa: F401
from test_gpu_rollout import _same_state
from test_gpu_tdm import compare_tdm_step, tdm_spawn

pytestmark = pytest.mark.gpu

CONTACT, TOUCH = 2, 4   # MACM_ENV_CONTACT_OVERFLOW, MACM_ENV_TOUCH_OVERFLOW
STEPS, CHUNK, POOL = 40, 8, 48


def _parking_min(N):
    """Smallest effective max_touching: a rollout parks 20 bytes per agent slot in the 24-byte entries of the stage."""
    slots = 128 if N > 64 else 64 if N > 32 else 32 if N > 16 else 16
    need = (20 * slots + 23) // 24
    return (need + 15) // 16 * 16


def _cases():
    out = []
    for G, APL in SHAPES:
        for kind in ("flock", "tdm"):
            out.append(dict(build="default", G=G, APL=APL, kind=kind, wide=False, N=RAGGED_N[(G, APL)]))
    for G, APL in SHAPES[3:]:
        for kind in ("flock", "tdm"):
            out.append(dict(build="default", G=G, APL=APL, kind=kind, wide=True, N=RAGGED_N[(G, APL)]))
    for G, APL in SHAPES[4:]:
        for kind in ("flock", "tdm"):
            out.append(dict(build="huge", G=G, APL=APL, kind=kind, wide=False, N=RAGGED_N[(G, APL)]))
    out.append(dict(build="huge", G=32, APL=4, kind="flock", wide=True, N=RAGGED_N[(32, 4)]))
    return out


CASES = _cases()


def _case_id(c):
    return "%s-%s-G%d-APL%d-%s-N%d" % (c["build"], c["kind"], c["G"], c["APL"], "wide" if c["wide"] else "narrow", c["N"])


def _pool(c, rng):
    """POOL spawns from a dense pile to a sparse world, their actions, and the oracle's per-step counts
    (peak live contacts, touching contacts at Collide), each [STEPS, POOL]."""
    from oracle import oracle
    N, kind = c["N"], c["kind"]
    pile = PILE[(kind, "huge" if c["build"] == "huge" else ("wide" if c["wide"] else "narrow"))][N]
    sides = np.linspace(0.7 * pile, 1.6 * pile if c["build"] == "huge" else max(2.5 * pile, 4.0), POOL)
    acts = rng.integers(0, 3, (STEPS, POOL, N, 4))
    if kind == "flock":
        acts[..., 3] = 0
        pos = sides[:, None, None] * (rng.random((POOL, N, 2)) - 0.5)
        ang = rng.uniform(-1, 1, (POOL, N)) * np.pi
        ta, td = 2 * np.pi * rng.random((POOL, 1)), 25 + rng.random((POOL, 1)) * 35
        spawn = dict(pos=pos, ang=ang, tg=np.stack([td * np.cos(ta), td * np.sin(ta)], -1))
        ref = oracle.OracleBatch(POOL, n_agents=N, n_targets=1, **oracle_kwargs(FLOCK_A))
        ref.reset(pos, ang, targets=spawn["tg"])
    else:
        acts[..., 3] = rng.random((STEPS, POOL, N)) < 0.9
        parts = [tdm_spawn(rng, 1, _teams(N), s, s) for s in sides]
        team = parts[0][0]
        spawn = dict(pos=np.concatenate([p[1] for p in parts]), ang=np.concatenate([p[2] for p in parts]), team=team)
        ref = oracle.OracleBatch(POOL, env_kind=oracle.TDM, n_agents=N, n_targets=0)
        ref.reset(spawn["pos"], spawn["ang"], team=team)
    live, touch = np.zeros((STEPS, POOL), int), np.zeros((STEPS, POOL), int)
    for k in range(STEPS):
        ref.flock_step(acts[k, ..., :3]) if kind == "flock" else ref.tdm_step(acts[k])
        for e in range(POOL):
            i = ref.env_info(e)
            live[k, e], touch[k, e] = i["peak_contacts"], i["touching"]
    return spawn, acts, live, touch


def _pick(counts, step, lo, hi, ok=lambda v: np.ones(POOL, bool)):
    """A capacity v (a multiple of `step` in [lo, hi]) that one pool env (among ok(v)) reaches exactly and another one
    exceeds: (v, at, over).  The over env is preferred to exceed by exactly one on its first step above v."""
    peak = counts.max(0)
    best = None
    for v in range(lo, hi + 1, step):
        at = [e for e in np.flatnonzero(ok(v)) if peak[e] == v]
        over = [e for e in np.flatnonzero(ok(v)) if peak[e] > v]
        if not at or not over:
            continue
        first = {e: counts[np.argmax(counts[:, e] > v), e] - v for e in over}
        o = min(over, key=lambda e: (first[e], peak[e]))
        score = (first[o], -len(over))
        if best is None or score < best[0]:
            best = (score, v, at[0], o)
    return None if best is None else best[1:]


def _batch(E, at, over, below):
    """Pool indices of the batch: the over env shares the first warp with the at env and is also the last env (a
    write past its rows lands beyond the buffers); envs below the capacity, densest first, fill the rest."""
    fill = list(below) or [at]
    idx = [fill[i % len(fill)] for i in range(E)]
    idx[1], idx[2], idx[E // 2], idx[E - 1] = over, at, at, over
    return np.array(idx)


def _guarded(engine, names, band=4096):
    """Rebind (macm_bind) the engine's buffers `names` as slices of larger allocations whose bands before and after
    hold a sentinel; returns a function that asserts the bands are intact."""
    import torch
    from gym_macm import _lib
    held = []
    for n in names:
        t = engine.t[n]
        nbytes = t.numel() * t.element_size()
        if nbytes == 0:
            continue
        raw = torch.full((nbytes + 2 * band,), 0xA5, dtype=torch.uint8, device=engine.device)
        view = raw[band:band + nbytes].view(t.dtype).view(t.shape)
        view.copy_(t)
        engine.t[n] = view
        held.append((n, raw, nbytes))
    bufs = _lib.MacmBuffers()
    for n, t in engine.t.items():
        setattr(bufs, n, t.data_ptr())
    _lib.check(_lib.lib().macm_bind(engine._h, C.byref(bufs)), engine._h)

    def check(k):
        for n, raw, nbytes in held:
            r = raw.cpu().numpy()
            assert (r[:band] == 0xA5).all() and (r[band + nbytes:] == 0xA5).all(), "step %d: write outside %s" % (k, n)
    return check


def _sims(c, E, spawn, idx, caps, n=2, **kw):
    import gym_macm
    from oracle import oracle
    N = c["N"]
    if c["kind"] == "flock":
        sims = [gym_macm.BatchedFlock(E, n_agents=[N], device="cuda:0", seed=None, **caps, **FLOCK_A, **kw)
                for _ in range(n)]
        for s in sims:
            s.load_state(spawn["pos"][idx], spawn["ang"][idx], targets=spawn["tg"][idx])
        ref = oracle.OracleBatch(E, n_agents=N, n_targets=1, **oracle_kwargs(dict(FLOCK_A, **kw)))
        ref.reset(spawn["pos"][idx], spawn["ang"][idx], targets=spawn["tg"][idx])
        return sims, ref
    sims = [gym_macm.BatchedTDM(E, n_agents=_teams(N), device="cuda:0", seed=None, **caps, **kw) for _ in range(n)]
    for s in sims:
        s.load_state(spawn["pos"][idx], spawn["ang"][idx])
    ref = oracle.OracleBatch(E, env_kind=oracle.TDM, n_agents=N, n_targets=0)
    ref.reset(spawn["pos"][idx], spawn["ang"][idx], team=spawn["team"])
    return sims, ref


def _hold(sim, ref, o, k, c, held):
    if c["kind"] == "flock":
        compare_step(sim, ref, o, k, envs=held)
    else:
        compare_tdm_step(sim, ref, o, k, contact_envs=None, envs=held)


def _run(c, what, spawn, acts, live, touch, guard=False):
    """Step a batch whose capacity for `what` ("contacts" / "touching") sits at the edge of its envs' counts."""
    import torch
    threads, E, mt_full = _launch(c)
    N, pairs = c["N"], c["N"] * (c["N"] - 1) // 2
    huge = c["build"] == "huge"
    if what == "contacts":
        # max_touching is capped at max_contacts; in the huge build a C above 240 keeps the global-memory stage
        if huge:
            teff = lambda v: (v + 15) // 16 * 16
        else:
            teff = lambda v: max(_parking_min(N), (min(mt_full, v) + 15) // 16 * 16)
        # envs whose touching counts stay within the touching capacity that comes with C = v
        pick = _pick(live, 1, 241 if huge else 1, pairs, lambda v: touch.max(0) <= teff(v))
        if pick is None:
            return None
        v, at, over = pick
        caps, want_t = dict(max_contacts=v, max_touching=mt_full), teff(v)
        below = [e for e in np.argsort(-live.max(0)) if touch[:, e].max() <= want_t and live[:, e].max() <= v]
    else:
        lo, step, hi = (256, 16, pairs) if huge else (_parking_min(N), 16, mt_full)
        pick = _pick(touch, step, lo, hi)
        if pick is None:
            return None
        v, at, over = pick
        caps, want_t = dict(max_contacts=pairs, max_touching=v), v
        below = [e for e in np.argsort(-touch.max(0)) if touch[:, e].max() <= v]
    idx = _batch(E, at, over, below)
    (one, roll), ref = _sims(c, E, spawn, idx, caps)
    info, sizes = one.engine.info, one.engine.sizes
    assert (info.lanes_per_env, info.agents_per_lane, info.threads_per_block) == (c["G"], c["APL"], threads)
    assert (sizes.touch_scratch > 0) == (c["build"] == "huge")
    Ceff, Teff = sizes.max_contacts, sizes.max_touching
    assert (Ceff, Teff) == (caps["max_contacts"], want_t), (Ceff, Teff, caps)
    check = _guarded(one.engine, ("contact_ab", "contact_imp", "touch_scratch")) if guard else None
    a = torch.as_tensor(acts[:, idx].astype(np.uint8), device="cuda:0")
    ever = np.zeros(E, int)           # the oracle's bits: count above capacity at some step so far
    prev = np.zeros(E, int)
    first = {}
    chunk_start = 0
    for k in range(STEPS):
        one.step(a[k])
        o = ref.flock_step(acts[k, idx, :, :3]) if c["kind"] == "flock" else ref.tdm_step(acts[k, idx])
        bits = overflow_bits(one, ref, prev, ever, k)
        for e in np.flatnonzero(bits & ~prev):
            first.setdefault(int(e), k)
        prev = bits
        held = bits == 0
        _hold(one, ref, o, k, c, held)
        if check:
            check(k)
        if k + 1 - chunk_start == CHUNK:
            roll.rollout(a[chunk_start:k + 1])
            torch.cuda.synchronize()
            _same_state(one, roll, "rollout up to step %d" % k)
            chunk_start = k + 1
    bit = CONTACT if what == "contacts" else TOUCH
    assert not (prev[idx == at] & bit).any(), "the env at the capacity was flagged"
    k_over = int(np.argmax((live if what == "contacts" else touch)[:, over] > v))
    assert first.get(E - 1) == k_over and prev[E - 1] & bit, (first, k_over)
    for s in (one, roll):
        s.close()
    return v, Teff, k_over


@pytest.mark.parametrize("c", CASES, ids=[_case_id(c) for c in CASES])
def test_capacity_edge(c, block_threads):
    threads, _, _ = _launch(c)
    block_threads(threads)
    rng = np.random.default_rng(500 + 1000 * c["G"] + 10 * c["APL"] + c["N"] + (7 if c["kind"] == "tdm" else 0))
    spawn, acts, live, touch = _pool(c, rng)
    guard = c["build"] == "huge" and not c["wide"]
    ran = [_run(c, what, spawn, acts, live, touch, guard=guard) for what in ("contacts", "touching")]
    assert ran[0] is not None, "no contact capacity with an env at it and one above it"
    # the touching capacity cannot be exceeded where N(N-1)/2 is below its smallest effective value
    if c["N"] * (c["N"] - 1) // 2 > 2 * _parking_min(c["N"]):
        assert ran[1] is not None, "no touching capacity with an env at it and one above it"


def _capacity_run_setup(c, what, rng):
    """(spawn, actions, batch pool indices, capacities, capacity value, its first step above it) of a case."""
    spawn, acts, live, touch = _pool(c, rng)
    N, pairs = c["N"], c["N"] * (c["N"] - 1) // 2
    counts = live if what == "contacts" else touch
    v, at, over = _pick(counts, 1, 1, pairs, lambda v: touch.max(0) <= 240) if what == "contacts" else \
        _pick(touch, 16, _parking_min(N), 240)
    below = [e for e in np.argsort(-counts.max(0)) if counts[:, e].max() <= v and touch[:, e].max() <= 240]
    caps = dict(max_contacts=v, max_touching=240) if what == "contacts" else dict(max_contacts=pairs, max_touching=v)
    return spawn, acts, below, at, over, caps, int(np.argmax(counts[:, over] > v))


def test_overflow_reset_final_rollout_and_check():
    """Flagged envs through the rest of the API: overflow_count() counts the bits, check_overflow raises on the first
    flagging step and not before, an auto-reset clears the bits while the finished episode's final env_state row keeps
    them, a rollout with auto-reset equals the single steps, and reset_done() gives a flagged env a new episode that
    is bit-exact again."""
    import torch
    import gym_macm
    from gym_macm import _lib
    c = dict(build="default", G=32, APL=2, kind="flock", wide=False, N=50)
    rng = np.random.default_rng(77)
    spawn, acts, below, at, over, caps, k_over = _capacity_run_setup(c, "contacts", rng)
    E, K, T = 12, 24, 16   # time_limit 0.25 s: done after step 16, when the auto-reset sims start new episodes
    assert 0 < k_over < T - 1   # "not before" means something, and the episode that ends carries the bit
    idx = np.array([below[i % len(below)] for i in range(E)])
    idx[[3, 4, E - 1]] = at, over, over
    (one,), ref = _sims(c, E, spawn, idx, caps, n=1, keep_final=True)
    auto, roll = _sims(c, E, spawn, idx, caps, n=2, keep_final=True, auto_reset=True, time_limit=0.25)[0]
    (chk,), _ = _sims(c, E, spawn, idx, caps, n=1, check_overflow=True)
    a = torch.as_tensor(acts[:K, idx].astype(np.uint8), device="cuda:0")
    out = roll.rollout(a, want=("obs", "nn_idx", "rewards", "collided", "done", "final_env_state"))
    per, bits_at = {n: [] for n in ("obs", "nn_idx", "rewards", "collided", "done")}, {}
    for k in range(K):
        one.step(a[k])
        auto.step(a[k])
        o = ref.flock_step(acts[k, idx, :, :3])
        torch.cuda.synchronize()
        bits = one.state["env_state"][:, 1].cpu().numpy() & (CONTACT | TOUCH)
        bits_at[k] = bits
        if k < k_over:
            chk.step(a[k])
        elif k == k_over:
            assert bits.any()
            with pytest.raises(_lib.MacmError):
                chk.step(a[k])
        assert one.overflow_count() == (int((bits & CONTACT).astype(bool).sum()), int((bits & TOUCH).astype(bool).sum()))
        compare_step(one, ref, o, k, envs=bits == 0)
        for n in per:
            per[n].append(auto.state[n].clone())
        abits = auto.state["env_state"][:, 1].cpu().numpy() & (CONTACT | TOUCH)
        if k == T - 1:
            assert auto.done.all() and not abits.any()
            assert (auto.episode.cpu().numpy() == 1).all()
            fin = auto.final_info
            assert np.array_equal(fin["overflowed"].cpu().numpy(), bits != 0)
            assert np.array_equal(auto.engine.final["env_state"][:, 1].cpu().numpy() & 6, bits)
        elif k < T - 1:
            assert np.array_equal(abits, bits)
    assert bits_at[K - 1][E - 1] and bits_at[K - 1][4] and not bits_at[K - 1][3]
    torch.cuda.synchronize()
    _same_state(auto, roll, "rollout with auto-reset")
    for n in per:
        assert torch.equal(out[n], torch.stack(per[n])), n
    assert torch.equal(out["final_env_state"][T - 1], auto.engine.final["env_state"])
    # reset_done on the flagged envs: bits cleared, the final row keeps them, the new episode is exact
    flagged = bits_at[K - 1] != 0
    one.reset_done(torch.as_tensor(flagged, device="cuda:0"), seed=5)
    torch.cuda.synchronize()
    assert not (one.state["env_state"][:, 1].cpu().numpy() & 6).any()
    assert np.array_equal(one.engine.final["env_state"][flagged, 1].cpu().numpy() & 6, bits_at[K - 1][flagged])
    pv = one.state["posvel"].cpu().numpy().astype(np.float64)
    ang = one.state["angsleep"][..., 0].cpu().numpy().astype(np.float64)
    tg = one.state["targets"].cpu().numpy().astype(np.float64)
    for e in np.flatnonzero(flagged):
        ref.reset_env(int(e), pv[e, :, 0:2], ang[e], tg[e])
    for k in range(8):
        act = rng.integers(0, 3, (E, c["N"], 3))
        one.step(torch.as_tensor(act, device="cuda:0"))
        compare_step(one, ref, ref.flock_step(act), K + k)
    for s in (one, auto, roll, chk):
        s.close()


def test_default_capacity_beyond_64_agents():
    """65..128 agents: the 192-contact shared stage (fourteen 128-agent envs to a wide block) with a global-memory stage
    of 3N behind it."""
    import gym_macm
    for N, want in ((65, 200), (100, 304), (128, 384)):
        env = gym_macm.BatchedFlock(2048, n_agents=[N], device="cuda:0", seed=1)
        assert env.engine.sizes.max_touching == want and env.engine.sizes.touch_scratch == 2048 * want * 32, N
        if N == 128:
            assert env.engine.info.envs_per_block == 14 and env.engine.info.threads_per_block == 448
        env.close()
    env = gym_macm.BatchedFlock(16, n_agents=[64], device="cuda:0", seed=1)
    assert (env.engine.sizes.max_touching, env.engine.sizes.touch_scratch) == (128, 0)
    env.close()


EPISODE = 3601   # steps of a default episode (time_limit 60 s at 60 Hz)


@pytest.mark.parametrize("N", [16, 32, 64, 100, 116, 128])
def test_gathered_flock_at_default_capacity(N):
    """The device's flock actor (bots.flock: head for the target) for a whole episode at the default capacities: the
    agents gather in a pile at the target, and no env may run out of contact capacity.  The oracle starts from the
    device's sampled state and gets the device's actions; it holds every env every 400 steps."""
    import torch
    import gym_macm
    from oracle import oracle
    E = 16
    env = gym_macm.BatchedFlock(E, n_agents=[N], device="cuda:0", seed=300 + N)
    torch.cuda.synchronize()
    pv = env.state["posvel"].cpu().numpy().astype(np.float64)
    ang = env.state["angsleep"][..., 0].cpu().numpy().astype(np.float64)
    ref = oracle.OracleBatch(E, n_agents=N, n_targets=1)
    ref.reset(pv[..., 0:2], ang, targets=env.state["targets"].cpu().numpy().astype(np.float64))
    most = 0
    for k in range(EPISODE):
        a = env.bot_actions("flock")
        env.step(a)
        o = ref.flock_step(a.cpu().numpy()[..., :3].astype(np.int64))
        most = max(most, max(ref.env_info(e)["touching"] for e in range(E)))
        if k % 400 == 399 or k == EPISODE - 1:
            compare_step(env, ref, o, k, check_contacts_envs=range(4))
    assert env.overflow_count() == (0, 0)
    assert bool(env.done.all())
    if N > 64:
        assert most > 1.4 * N, most   # the flock did gather
    env.close()


@pytest.mark.parametrize("teams", [[15, 15, 15], [64, 64]], ids=["3x15", "2x64"])
def test_combat_bots_at_default_capacity(teams):
    """TDM with every agent driven by the device's combat actor (bots.combat: face, approach and strike the nearest
    enemy) at the default capacities, held to the oracle until the episode ends."""
    import torch
    import gym_macm
    from oracle import oracle
    E, N = 8 if len(teams) == 3 else 4, sum(teams)
    env = gym_macm.BatchedTDM(E, n_agents=teams, device="cuda:0", seed=400 + N)
    torch.cuda.synchronize()
    pv = env.state["posvel"].cpu().numpy().astype(np.float64)
    ang = env.state["angsleep"][..., 0].cpu().numpy().astype(np.float64)
    team = np.array([t for t, n in enumerate(teams) for _ in range(n)], np.uint8)
    ref = oracle.OracleBatch(E, env_kind=oracle.TDM, n_agents=N, n_targets=0)
    ref.reset(pv[..., 0:2], ang, team=team)
    for k in range(EPISODE):
        a = env.bot_actions("combat", seed=k)
        env.step(a)
        o = ref.tdm_step(a.cpu().numpy().astype(np.int64))
        if k % 400 == 399 or k == EPISODE - 1:
            compare_tdm_step(env, ref, o, k, contact_envs=4)
    assert env.overflow_count() == (0, 0)
    env.close()
