"""Batched tensor API over libmacm.so: thousands of independent Flock worlds stepped by one kernel.

`BatchedFlock` keeps the reference's surface -- `obs`, `agents`, `done`, `targets`, `settings`,
`step(actions) -> (obs, rewards)` (gym_macm/envs/mvmnt.py:35-140) -- with torch CUDA tensors
where the reference has per-agent Python objects.  All simulator state lives in caller-owned
torch tensors (SoA, env-major) that the C ABI reads and writes in place; this module does no
arithmetic of its own and has no CPU path.
"""
import ctypes as C

import numpy as np

from . import _lib
from .settings import combatSettings, flockSettings


def _torch():
    import torch
    return torch


def _as_list(n_agents):
    # the reference wants a list (mvmnt.py:61 `sum(self.n_agents)`); README.md:44 passes an int (App. B4)
    if isinstance(n_agents, (int, np.integer)):
        return [int(n_agents)]
    return [int(x) for x in n_agents]


def flock_params(settings, n_envs, n_agents, n_targets):
    """flockSettings -> macm_params (field-by-field; file:line in include/macm.h)."""
    p = _lib.default_params(_lib.FLOCK)
    fx = settings.bodySettings["fixtures"]
    p.n_envs, p.n_agents, p.n_targets = int(n_envs), int(n_agents), int(n_targets)
    p.max_contacts, p.max_touching = int(settings.max_contacts), int(settings.max_touching)
    p.hz = float(settings.hz)
    p.velocity_iterations = int(settings.velocityIterations)
    p.position_iterations = int(settings.positionIterations)
    p.warm_starting = int(bool(settings.enableWarmStarting))
    p.damping_model = _lib.DAMPING[str(settings.damping_model)]
    p.radius, p.density, p.friction = float(fx.radius), float(fx.density), float(fx.friction)
    p.linear_damping = float(settings.bodySettings["linearDamping"])
    p.agent_force = float(settings.agent_force)
    p.agent_rotation_speed = float(settings.agent_rotation_speed)
    p.time_limit = float(settings.time_limit)
    p.reward_mode = _lib.REWARD[settings.reward_mode]
    p.action_mode = _lib.ACTION[settings.action_mode]
    p.coord = _lib.COORD[settings.coord]
    p.reward_radius = float(settings.reward_radius)
    p.start_spread = float(settings.start_spread)
    p.start_x, p.start_y = float(settings.start_point[0]), float(settings.start_point[1])
    p.target_mindist, p.target_maxdist = float(settings.target_mindist), float(settings.target_maxdist)
    p.env_index_base = int(settings.env_index_base)
    if settings.auto_reset:
        p.flags |= _lib.FLAG_AUTO_RESET
    return p


def tdm_params(settings, n_envs, n_agents):
    """combatSettings (+ combat.Agent constants) -> macm_params."""
    p = _lib.default_params(_lib.TDM)
    fx = settings.bodySettings["fixtures"]
    p.n_envs, p.n_agents, p.n_targets = int(n_envs), int(n_agents), 0
    p.max_contacts, p.max_touching = int(settings.max_contacts), int(settings.max_touching)
    p.hz = float(settings.hz)
    p.velocity_iterations = int(settings.velocityIterations)
    p.position_iterations = int(settings.positionIterations)
    p.warm_starting = int(bool(settings.enableWarmStarting))
    p.damping_model = _lib.DAMPING[str(settings.damping_model)]
    p.radius, p.density, p.friction = float(fx.radius), float(fx.density), float(fx.friction)
    p.linear_damping = float(settings.bodySettings["linearDamping"])
    p.agent_force = float(settings.agent_force)
    p.agent_rotation_speed = float(settings.agent_rotation_speed)
    p.time_limit = float(settings.time_limit)
    p.flags = (_lib.FLAG_REPAIR_MOV_COOLDOWN if settings.repair_mov_cooldown else 0) | \
              (_lib.FLAG_AUTO_RESET if settings.auto_reset else 0)
    p.cooldown_atk, p.cooldown_mov_penalty = float(settings.cooldown_atk), float(settings.cooldown_mov_penalty)
    p.melee_range, p.melee_dmg = float(settings.melee_range), float(settings.melee_dmg)
    p.percent_mov_penalty, p.init_health = float(settings.percent_mov_penalty), float(settings.init_health)
    p.world_width, p.world_height = float(settings.world_width), float(settings.world_height)
    p.env_index_base = int(settings.env_index_base)
    return p


class Engine(object):
    """A macm_sim handle plus the torch tensors bound to it."""

    OUTPUTS = ("obs", "rewards", "done", "nn_idx", "collided")   # order inside the output slab

    _DTYPES = dict(posvel="float32", angsleep="float32", fat="float32", contact_ab="int32", contact_imp="float32",
                   contact_count="int32", env_state="int32", targets="float32", target_idx="uint8",
                   tdm_state="float32", team="uint8", obs="float32", nn_idx="int32", rewards="float32",
                   collided="uint8", done="uint8", touch_scratch="uint8")

    def __init__(self, params, device=None):
        torch = _torch()
        self._h = None
        self._pinned = None
        L = _lib.lib()  # raises when libmacm.so has not been built
        if not torch.cuda.is_available():
            raise _lib.MacmError("gym_macm needs a CUDA device: the simulator is CUDA-only and has no CPU fallback")
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if self.device.type != "cuda":
            raise _lib.MacmError("gym_macm needs a CUDA device, got %r" % (self.device,))
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.params = params
        h = C.c_void_p()
        with torch.cuda.device(self.device):
            torch.cuda.init()
            rc = L.macm_create(C.byref(h), C.byref(params), self.device.index)
        if rc != 0:   # a handle returned with an error only carries the CUDA error text
            try:
                _lib.check(rc, h if h else None)
            finally:
                if h:
                    L.macm_destroy(h)
        self._h = h
        self.sizes = _lib.MacmBufferSizes()
        _lib.check(L.macm_get_buffer_sizes(h, C.byref(self.sizes)))
        self.info = _lib.MacmLaunchInfo()
        _lib.check(L.macm_get_launch_info(h, C.byref(self.info)))
        E, N, T = params.n_envs, params.n_agents, params.n_targets
        Cc, D = self.sizes.max_contacts, self.sizes.obs_dim
        shapes = dict(posvel=(E, N, 4), angsleep=(E, N, 2), fat=(E, N, 4), contact_ab=(E, Cc), contact_imp=(E, Cc, 2),
                      contact_count=(E,), env_state=(E, 4), targets=(E, T, 2), target_idx=(N,), tdm_state=(E, N, 4),
                      team=(N,), obs=(E, N, D), nn_idx=(E, N), rewards=(E, N), collided=(E, N), done=(E,),
                      touch_scratch=(int(self.sizes.touch_scratch),))
        self.t = {}
        bufs = _lib.MacmBuffers()
        # The per-step outputs live back to back in ONE device slab (each array 16-byte aligned), in the order
        # a learner asks for them; the pinned host mirror (pinned()) has the same layout, so macm_step_host moves
        # a step's results in a single device->host transfer.
        self._out_layout, off = {}, 0
        for name in self.OUTPUTS:
            nbytes = getattr(self.sizes, name)
            if nbytes:
                self._out_layout[name] = (off, nbytes)
                off = (off + nbytes + 15) // 16 * 16
        self._out_bytes = off
        slab = torch.zeros(off, dtype=torch.uint8, device=self.device)
        self._out_slab = slab
        for name in _lib.BUFFER_NAMES:
            nbytes = getattr(self.sizes, name)
            if nbytes == 0:
                continue
            dt = getattr(torch, self._DTYPES[name])
            if name in self._out_layout:
                o = self._out_layout[name][0]
                ten = slab[o:o + nbytes].view(dt).view(shapes[name])
            else:
                ten = torch.zeros(shapes[name], dtype=dt, device=self.device)
            assert ten.numel() * ten.element_size() == nbytes, (name, ten.shape, nbytes)
            self.t[name] = ten
            setattr(bufs, name, ten.data_ptr())
        _lib.check(L.macm_bind(h, C.byref(bufs)), h)
        self.E, self.N, self.T, self.C, self.obs_dim = E, N, T, Cc, D
        self.action_bytes = self.sizes.action_bytes
        self.final = None

    def bind_final(self):
        """Allocate and bind (macm_bind_final) the final arrays: obs, env_state and nn_idx (Flock) / tdm_state (TDM),
        shaped like the bound buffers of the same names.  Every reset copies the env's rows there first, so after a
        reset `final` holds the finished episode's terminal observation and outcome; rows of envs that were never
        reset keep their zeros."""
        torch = _torch()
        self.final = {n: torch.zeros_like(self.t[n]) for n in _lib.FINAL_NAMES if n in self.t}
        f = _lib.MacmFinalOut()
        for n, ten in self.final.items():
            setattr(f, n, ten.data_ptr())
        _lib.check(_lib.lib().macm_bind_final(self._h, C.byref(f)), self._h)
        return self.final

    def close(self):
        h, self._h = self._h, None
        if h:
            _lib.lib().macm_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    stream = None   # a torch.cuda.Stream this engine enqueues on; None = torch's current stream at call time

    def _stream(self, stream=None):
        stream = stream if stream is not None else self.stream
        if stream is not None:
            return C.c_void_p(stream.cuda_stream)
        return C.c_void_p(_torch().cuda.current_stream(self.device).cuda_stream)

    def reset(self):
        _lib.check(_lib.lib().macm_reset(self._h, self._stream()), self._h)

    def sample_reset(self, seed):
        _lib.check(_lib.lib().macm_sample_reset(self._h, C.c_uint64(int(seed) & (2 ** 64 - 1)), self._stream()), self._h)

    def reset_masked(self, mask=None, seed=0, stream=None):
        """macm_reset_masked: a new episode for the envs whose `mask` entry (uint8 / bool [E], device) is set;
        mask=None selects the envs whose `done` flag is set."""
        ptr = None
        if mask is not None:
            torch = _torch()
            if mask.dtype == torch.bool:
                mask = mask.to(torch.uint8)
            mask = mask.to(self.device).contiguous()
            assert mask.dtype == torch.uint8 and mask.numel() == self.E
            ptr = C.c_void_p(mask.data_ptr())
        _lib.check(_lib.lib().macm_reset_masked(self._h, ptr, C.c_uint64(int(seed) & (2 ** 64 - 1)), self._stream(stream)),
                   self._h)

    def set_auto_reset_seed(self, seed):
        _lib.check(_lib.lib().macm_set_auto_reset_seed(self._h, C.c_uint64(int(seed) & (2 ** 64 - 1))), self._h)

    def overflow_count(self):
        """(envs with dropped contacts, envs whose solver stage overflowed) -- synchronises the stream."""
        a, b = C.c_int32(0), C.c_int32(0)
        _lib.check(_lib.lib().macm_overflow_count(self._h, C.byref(a), C.byref(b), self._stream()), self._h)
        return int(a.value), int(b.value)

    def pack_actions(self, src, out):
        """Integer tensor [E,N,3|4] on the device -> uint8 [E,N,4] action words (one small kernel of the library)."""
        src = src.contiguous()
        _lib.check(_lib.lib().macm_pack_actions(self._h, C.c_void_p(src.data_ptr()), int(src.element_size()),
                                                int(src.shape[-1]), C.c_void_p(out.data_ptr()), self._stream()), self._h)
        return out

    def step(self, actions, stream=None):
        """One step on torch's current stream, or on `stream` (a torch.cuda.Stream): independent batches stepped
        on different streams overlap on the device."""
        _lib.check(_lib.lib().macm_step(self._h, C.c_void_p(actions.data_ptr()), self._stream(stream)), self._h)

    def rollout(self, actions, n_steps, policy=None, seed=0, out=None, stream=None):
        """macm_rollout: `n_steps` steps in one launch.  `actions` is a device tensor with a leading step
        axis, or None with `policy` = a _lib.BOTS code (the actions=None mode).  `out` maps any of
        obs / nn_idx / rewards / collided / done / final_obs / final_nn_idx / final_tdm_state / final_env_state to a
        device tensor with a leading step axis (final_*: only rows of envs reset after that step are written)."""
        ro = _lib.MacmRolloutOut()
        for name, ten in (out or {}).items():
            setattr(ro, name, ten.data_ptr())
        ptr = C.c_void_p(actions.data_ptr()) if actions is not None else None
        _lib.check(_lib.lib().macm_rollout(self._h, ptr, int(n_steps), -1 if policy is None else int(policy),
                                           C.c_uint64(int(seed) & (2 ** 64 - 1)), C.byref(ro), self._stream(stream)), self._h)

    def rollout_buffers(self, n_steps, want=("obs", "nn_idx", "rewards", "collided", "done")):
        """Device tensors for the per-step outputs of rollout(): the bound output buffers with a leading step axis.
        final_obs / final_nn_idx / final_tdm_state / final_env_state have the shapes of obs / nn_idx / tdm_state /
        env_state; row [k][e] is only defined where env e was reset after step k (auto_reset and done[k][e])."""
        torch = _torch()
        base = lambda n: n[len("final_"):] if n.startswith("final_") else n
        return {n: torch.empty((int(n_steps),) + tuple(self.t[base(n)].shape), dtype=self.t[base(n)].dtype,
                               device=self.device)
                for n in want if base(n) in self.t and (n == base(n) or base(n) in _lib.FINAL_NAMES)}

    def observe(self):
        _lib.check(_lib.lib().macm_observe(self._h, self._stream()), self._h)

    def bot_actions(self, policy, seed, out):
        _lib.check(_lib.lib().macm_bot_actions(self._h, int(policy), C.c_uint64(int(seed) & (2 ** 64 - 1)),
                                               C.c_void_p(out.data_ptr()), self._stream()), self._h)

    def pinned(self):
        """Pinned host mirrors of the action input and of every per-step output (for step_host)."""
        if self._pinned is None:
            torch = _torch()
            adt = torch.uint8 if self.action_bytes == 4 else torch.float32
            ashape = (self.E, self.N, 4) if self.action_bytes == 4 else (self.E, self.N, 2)
            p = dict(actions=torch.zeros(ashape, dtype=adt).pin_memory())
            slab = torch.zeros(self._out_bytes, dtype=torch.uint8).pin_memory()   # same layout as the device slab
            p["_slab"] = slab
            for name, (o, nbytes) in self._out_layout.items():
                p[name] = slab[o:o + nbytes].view(self.t[name].dtype).view(self.t[name].shape)
            self._pinned = p
        return self._pinned

    def step_host(self, actions_host, want=("obs", "rewards", "nn_idx", "collided", "done"), wait=True):
        """macm_step_host: host actions in, host outputs out; the copies are part of the call.
        wait=False enqueues on the handle's stream (macm_step_host_async); call host_sync() before
        reading the returned pinned tensors."""
        p = self.pinned()
        src = actions_host
        if not (src.is_pinned() and src.is_contiguous()):   # pageable memory: stage it in the pinned mirror
            p["actions"].copy_(actions_host)
            src = p["actions"]
        ptr = lambda n: C.c_void_p(p[n].data_ptr()) if (n in want and n in p) else None
        fn = _lib.lib().macm_step_host if wait else _lib.lib().macm_step_host_async
        _lib.check(fn(self._h, C.c_void_p(src.data_ptr()), ptr("obs"), ptr("rewards"),
                      ptr("nn_idx"), ptr("collided"), ptr("done")), self._h)
        return p

    def host_sync(self):
        _lib.check(_lib.lib().macm_host_sync(self._h), self._h)

    @property
    def launch_count(self):
        return int(_lib.lib().macm_launch_count(self._h))


class _BatchedCommon(object):
    """What BatchedFlock and BatchedTDM share: episode bookkeeping, overflow reporting, renderer export."""

    @property
    def episode(self):
        """How many times each env has been reset by reset_done / auto_reset (int32 [E])."""
        return self.engine.t["env_state"][:, 1] >> _lib.ENV_EPISODE_SHIFT

    @property
    def overflowed(self):
        """bool [E]: the env ran out of contact capacity (`max_contacts`: newest pairs dropped; `max_touching`: the
        solver skipped the excess) at some step since its last reset -- from that step on its results differ from the
        reference's.  Sticky until the env is reset.  `max_touching` up to 240 is a shared-memory stage; a larger value
        (up to `max_contacts`), and the default beyond 64 agents, add a global-memory stage that takes the denser env
        exactly (gathered flocks, spawn piles)."""
        return (self.engine.t["env_state"][:, 1] & (_lib.ENV_CONTACT_OVERFLOW | _lib.ENV_TOUCH_OVERFLOW)) != 0

    def overflow_count(self):
        """(envs with dropped contacts, envs with a truncated solver stage); one small kernel + a 8-byte read."""
        return self.engine.overflow_count()

    def _check_overflow(self):
        if self.settings.check_overflow:
            c, t = self.engine.overflow_count()
            if c or t:
                raise _lib.MacmError("contact capacity overflow: %d envs dropped contacts (max_contacts=%d), %d envs "
                                     "exceeded the solver stage (max_touching=%d); results of those envs "
                                     "differ from the reference's" % (c, self.engine.C, t, self.engine.sizes.max_touching))

    def _final(self):
        if self.engine.final is None:
            raise _lib.MacmError("final_obs / final_info need keep_final=True")
        return self.engine.final

    @property
    def final_info(self):
        """The outcome of each env's last finished episode, from the env state a reset copies before it overwrites it
        (keep_final=True): step_count, episode and overflowed, plus winner for TDM, each [E].  A row is valid where
        `done` is set after an auto-reset step, or where a reset_done mask was set; other rows hold an earlier
        episode's values (zeros before the first reset)."""
        es = self._final()["env_state"]
        info = {"step_count": es[:, 0], "episode": es[:, 1] >> _lib.ENV_EPISODE_SHIFT,
                "overflowed": (es[:, 1] & (_lib.ENV_CONTACT_OVERFLOW | _lib.ENV_TOUCH_OVERFLOW)) != 0}
        if self.engine.params.env_kind == _lib.TDM:
            info["winner"] = es[:, 3]
        return info

    def reset_done(self, mask=None, seed=0):
        """The reference's env.reset() (mvmnt.py:224-233, combat.py:229-239) for SOME envs of the batch: those
        whose `mask` entry is set, or with mask=None those that are done (time limit, mvmnt.py:134-136; one team
        left, combat.py:171-182).  Fresh states drawn on the device, keyed by (seed, env, agent, episode)."""
        self.engine.reset_masked(mask, seed)
        return self.obs

    def render_state(self, env=0):
        """One env of the batch as the objects the reference's CPU renderer reads
        (backends/pyglet_framework.py:122-180: `body.transform`, `body.userData.color`, fixtures' circle shape;
        `gui_objects` as filled by mvmnt.py:54-57): see gym_macm.render.  A device->host read of ~1 KB."""
        from gym_macm import render
        return render.export(self, int(env))


class BatchPool(object):
    """Several independent batches stepped round-robin, each on one of `n_streams` CUDA streams of its own.

    One batch of a few thousand envs is a single wave of blocks: the launch ends when its slowest env does (a few
    worlds with long contact islands), and a dependent launch can only start then.  A rollout worker normally holds
    several independent batches (double/triple buffering against the learner); giving consecutive batches different
    streams lets the next batch's blocks take over each SM as the previous batch's block retires -- 18.8 instead of
    22.8 us per 4096 x 64 step on a B200 (profiles/README.md).  Results are bit-identical to serial stepping
    (tests/test_gpu_api.py::test_batches_on_their_own_streams).

        pool = BatchPool([BatchedFlock(4096, n_agents=[64], device=dev, seed=s) for s in range(4)])
        for k in range(steps):
            env = pool.step(actions[k])        # steps batch k % len(pool) on its stream; returns that batch
        pool.synchronize()
    """

    def __init__(self, batches, n_streams=2):
        torch = _torch()
        self.batches = list(batches)
        dev = self.batches[0].device
        cur = torch.cuda.current_stream(dev)
        self.streams = [torch.cuda.Stream(device=dev) for _ in range(max(1, min(int(n_streams), len(self.batches))))]
        for st in self.streams:
            st.wait_stream(cur)               # the batches were built on the current stream
        for k, b in enumerate(self.batches):
            b.engine.stream = self.streams[k % len(self.streams)]
        self.k = 0

    def __len__(self):
        return len(self.batches)

    def step(self, actions):
        """Step the next batch of the rotation with `actions` (the packed uint8 [E,N,4] / float32 [E,N,2] wire
        format, on the device); returns that batch (its tensors are valid on its stream)."""
        b = self.batches[self.k % len(self.batches)]
        self.k += 1
        b.engine.step(actions)
        return b

    def stream_of(self, batch_index):
        return self.batches[batch_index % len(self.batches)].engine.stream

    def synchronize(self):
        for st in self.streams:
            st.synchronize()


class BatchedFlock(_BatchedCommon):
    """E independent Flock environments (gym_macm/envs/mvmnt.py) on one GPU.

    Same constructor keywords as the reference (`n_agents`, `actors`, `colors`, `targets`, any
    flockSettings attribute) plus `n_envs`, `device`, `seed`.  `obs` keeps the reference's dict
    keys with tensor values:

        obs["nodes"][0] = {"type": 0, "id": int32 [E,N],  "position": float32 [E,N,2|3]}   nearest agent
        obs["nodes"][1] = {"type": 1, "id": N,            "position": float32 [E,N,2|3]}   target

    `step(actions)` takes uint8 [E,N,4] (a0,a1,a2,pad) or any integer tensor [E,N,3] on the device
    (continuous mode: float32 [E,N,2]) and returns `(obs, rewards)` with rewards float32 [E,N].
    """

    name = "Flock v0 (batched)"

    def __init__(self, n_envs, n_agents=[10], actors=None, colors=None, targets=None, device=None, seed=0, stream=None,
                 **kwargs):
        self.settings = flockSettings(**kwargs)
        self.n_agents = _as_list(n_agents)
        self.n_envs = int(n_envs)
        N = sum(self.n_agents)
        self.n_targets = 1 if targets is None else len(np.unique(targets))
        # App. B4 repaired: default covers every agent, not just n_agents[0] of them
        self.targets_idx = [0] * N if targets is None else [int(t) for t in targets]
        if len(self.targets_idx) != N:
            raise ValueError("targets must name a target for each of the %d agents" % N)
        uniq = sorted(set(self.targets_idx))
        if uniq != list(range(len(uniq))):
            raise ValueError("targets must use the indices 0..T-1")
        self.actors, self.colors = actors, colors
        self.engine = Engine(flock_params(self.settings, self.n_envs, N, self.n_targets), device)
        if self.settings.keep_final:
            self.engine.bind_final()
        # Independent batches given a stream each overlap on the device (one batch's last envs finish while the
        # next batch starts); with stream=None every call goes to torch's current stream.
        self.engine.stream = stream
        torch = _torch()
        self.engine.t["target_idx"].copy_(torch.tensor(self.targets_idx, dtype=torch.uint8))
        self.agents = list(range(N))
        self._act4 = None
        if stream is not None:   # the buffers were allocated and filled on torch's current stream
            stream.wait_stream(torch.cuda.current_stream(self.device))
        if seed is not None:   # seed=None: the caller loads a state itself (load_state)
            self.reset(seed)

    # -- state ---------------------------------------------------------------------------------
    @property
    def device(self):
        return self.engine.device

    @property
    def state(self):
        """The live state tensors (views, not copies)."""
        return self.engine.t

    @property
    def targets(self):
        return self.engine.t["targets"]

    @property
    def done(self):
        return self.engine.t["done"].bool()

    @property
    def step_count(self):
        return self.engine.t["env_state"][:, 0]

    @property
    def time_passed(self):
        return self.step_count.double() * (1.0 / self.settings.hz)

    def reset(self, seed=0):
        """Fresh worlds with states drawn on the device from the reference's distributions
        (mvmnt.py:48-52,62-64).  (The reference's own reset() is broken, SURVEY App. B3.)"""
        self.engine.sample_reset(seed)
        return self.obs

    def load_state(self, pos, angle, vel=None, targets=None):
        """Create fresh worlds at given positions/angles, like a new b2World with bodies at
        `pos` (mvmnt.py:70-75): fat AABBs = tight +- 0.1, no contacts, first-step flags."""
        torch = _torch()
        t = self.engine.t
        E, N = self.engine.E, self.engine.N
        pos = torch.as_tensor(pos, dtype=torch.float32).reshape(E, N, 2)
        t["posvel"][..., 0:2] = pos.to(self.device)
        t["posvel"][..., 2:4] = 0 if vel is None else torch.as_tensor(vel, dtype=torch.float32).reshape(E, N, 2).to(self.device)
        t["angsleep"][..., 0] = torch.as_tensor(angle, dtype=torch.float32).reshape(E, N).to(self.device)
        if targets is not None:
            t["targets"].copy_(torch.as_tensor(targets, dtype=torch.float32).reshape(E, self.engine.T, 2))
        self.engine.reset()
        return self.obs

    # -- stepping ------------------------------------------------------------------------------
    @property
    def obs(self):
        o, D = self.engine.t["obs"], self.engine.obs_dim // 2
        return {"nodes": [{"type": 0, "id": self.engine.t["nn_idx"], "position": o[..., 0:D]},
                          {"type": 1, "id": self.engine.N, "position": o[..., D:2 * D]}]}

    @property
    def final_obs(self):
        """The terminal observation of each env's last finished episode (keep_final=True), laid out as `obs`: what
        `obs` held when the env was last reset (valid rows: see final_info)."""
        f, D = self._final(), self.engine.obs_dim // 2
        return {"nodes": [{"type": 0, "id": f["nn_idx"], "position": f["obs"][..., 0:D]},
                          {"type": 1, "id": self.engine.N, "position": f["obs"][..., D:2 * D]}]}

    @property
    def rewards(self):
        return self.engine.t["rewards"]

    @property
    def collided(self):
        return self.engine.t["collided"].bool()

    def pack_actions(self, actions):
        """Any integer tensor [E,N,3] -> the uint8 [E,N,4] wire format."""
        torch = _torch()
        E, N = self.engine.E, self.engine.N
        if self._act4 is None:
            self._act4 = torch.zeros((E, N, 4), dtype=torch.uint8, device=self.device)
        a = torch.as_tensor(actions, device=self.device)
        if a.dtype.is_floating_point or a.dtype == torch.bool:
            a = a.to(torch.uint8)
        return self.engine.pack_actions(a.reshape(E, N, -1), self._act4)

    def step(self, actions):
        torch = _torch()
        E, N = self.engine.E, self.engine.N
        if self.settings.action_mode == "discrete":
            a = actions
            if not (torch.is_tensor(a) and a.dtype == torch.uint8 and a.is_cuda and tuple(a.shape) == (E, N, 4)
                    and a.is_contiguous()):
                a = self.pack_actions(a)
        else:
            a = torch.as_tensor(actions, dtype=torch.float32, device=self.device).reshape(E, N, 2).contiguous()
        self.engine.step(a)
        self._check_overflow()
        return self.obs, self.engine.t["rewards"]

    def rollout(self, actions=None, n_steps=None, policy="random", seed=0, want=("obs", "nn_idx", "rewards", "collided", "done"),
                out=None):
        """`n_steps` consecutive steps in one kernel launch (macm_rollout) -- the reference's
        `for _ in range(n_steps): obs, rewards = env.step(a_k)` loop (README.md:8-14) with every env's bodies
        held on chip between its steps; bit-identical to calling step() n_steps times.

        actions: uint8 [K,E,N,4] on the device (continuous mode: float32 [K,E,N,2]), or None for the
        reference's actions=None mode (mvmnt.py:86-92) with every agent driven by the scripted actor `policy`
        (test_scripts/bots.py).  Returns a dict of per-step tensors (leading axis K) for the names in `want`;
        with "obs" left out the observation pass only runs after the last step (action repeat).  The usual
        attributes (obs, rewards, done, state) hold the last step's values afterwards.  With auto_reset, `want` may
        also name final_obs / final_nn_idx (Flock) / final_tdm_state (TDM) / final_env_state: the terminal rows of the
        envs reset after each step; only rows [k][e] with done[k][e] set are defined, the others are left as
        allocated (torch.empty)."""
        torch = _torch()
        E, N = self.engine.E, self.engine.N
        if actions is not None:
            a = actions
            if self.settings.action_mode == "discrete":
                if not (torch.is_tensor(a) and a.dtype == torch.uint8 and a.is_cuda and a.dim() == 4 and
                        tuple(a.shape[1:]) == (E, N, 4) and a.is_contiguous()):
                    a3 = torch.as_tensor(a, device=self.device)
                    a = torch.zeros((a3.shape[0], E, N, 4), dtype=torch.uint8, device=self.device)
                    a[..., 0:a3.shape[-1]] = a3.reshape(a3.shape[0], E, N, -1)
            else:
                a = torch.as_tensor(a, dtype=torch.float32, device=self.device).reshape(-1, E, N, 2).contiguous()
            K = int(a.shape[0]) if n_steps is None else int(n_steps)
            if K > a.shape[0]:
                raise ValueError("n_steps exceeds the leading axis of actions")
            pol = None
        else:
            if n_steps is None:
                raise ValueError("n_steps is required with actions=None")
            a, K, pol = None, int(n_steps), _lib.BOTS[policy]
        if out is None:
            out = self.engine.rollout_buffers(K, want)
        self.engine.rollout(a, K, pol, seed, out)
        self._check_overflow()
        return out

    def step_host(self, actions):
        """Same step through the host-buffer entry point (macm_step_host): `actions` is a CPU
        uint8 [E,N,4] / float32 [E,N,2] tensor; returns pinned CPU tensors."""
        p = self.engine.step_host(actions)
        D = self.engine.obs_dim // 2
        obs = {"nodes": [{"type": 0, "id": p["nn_idx"], "position": p["obs"][..., 0:D]},
                         {"type": 1, "id": self.engine.N, "position": p["obs"][..., D:2 * D]}]}
        return obs, p["rewards"]

    def bot_actions(self, policy="flock", seed=0, out=None):
        """test_scripts/bots.py on the device: one action per agent from the current obs."""
        torch = _torch()
        if out is None:
            out = torch.empty((self.engine.E, self.engine.N, 4), dtype=torch.uint8, device=self.device)
        self.engine.bot_actions(_lib.BOTS[policy], seed, out)
        return out

    def contacts(self, env):
        """Contact list of one env in birth order: (ab [n,2], touching [n], impulses [n,2]) on the CPU."""
        t = self.engine.t
        n = int(t["contact_count"][env])
        ab = t["contact_ab"][env, :n].cpu().numpy().astype(np.uint32)
        imp = t["contact_imp"][env, :n].cpu().numpy()
        return np.stack([ab & 0xff, (ab >> 8) & 0xff], -1).astype(np.int32), ((ab >> 16) & 1).astype(np.uint8), imp

    def close(self):
        self.engine.close()


class BatchedTDM(_BatchedCommon):
    """E independent team-deathmatch environments (gym_macm/envs/combat.py) on one GPU, with the
    repaired semantics of SURVEY.md Appendix B (the reference class cannot be constructed as
    shipped).  `n_agents=[15, 15, 15]` gives three teams; agent index = team-major order, the
    reference's ids are `str(team) + str(j)` (combat.py:87).

        obs = {"myHealth": float32 [E,N], "myTeam": uint8 [N], "alive": bool [E,N],
               "agents": {"type": float32 [E,N,N] (1 ally, 0 enemy, -1 no entry),
                          "position": float32 [E,N,N,3] = r, theta, phi}}       (combat.py:211-226)

    `step(actions)`: uint8 [E,N,4] = a0, a1, a2, attack (or any integer tensor of that shape);
    returns `(obs, rewards)`; rewards are -1 for an alive agent listed in a contact, else 0 (B12).
    """

    name = "Team Deathmatch (batched)"

    def __init__(self, n_envs, n_agents=[1, 1], actors=None, colors=None, device=None, seed=0, stream=None, **kwargs):
        self.settings = combatSettings(**kwargs)
        self.n_agents = _as_list(n_agents)
        self.n_envs = int(n_envs)
        self.teams = [t for t, n in enumerate(self.n_agents) for _ in range(n)]
        self.ids = [str(t) + str(j) for t, n in enumerate(self.n_agents) for j in range(n)]
        N = len(self.teams)
        if len(self.n_agents) > 8:
            raise ValueError("at most 8 teams")
        self.actors, self.colors = actors, colors
        self.engine = Engine(tdm_params(self.settings, self.n_envs, N), device)
        if self.settings.keep_final:
            self.engine.bind_final()
        self.engine.stream = stream
        torch = _torch()
        self.engine.t["team"].copy_(torch.tensor(self.teams, dtype=torch.uint8))
        self.agents = list(range(N))
        self._act4 = None
        if stream is not None:
            stream.wait_stream(torch.cuda.current_stream(self.device))
        if seed is not None:
            self.reset(seed)

    @property
    def device(self):
        return self.engine.device

    @property
    def state(self):
        return self.engine.t

    @property
    def done(self):
        return self.engine.t["done"].bool()

    @property
    def winner(self):
        return self.engine.t["env_state"][:, 3]

    @property
    def step_count(self):
        return self.engine.t["env_state"][:, 0]

    @property
    def alive(self):
        return (self.engine.t["tdm_state"][..., 3].view(_torch().int32) & 1).bool()

    @property
    def health(self):
        return self.engine.t["tdm_state"][..., 0]

    @property
    def cooldowns(self):
        """(attack, movement-penalty) cool-downs as whole steps left."""
        ts = self.engine.t["tdm_state"].view(_torch().int32)
        return ts[..., 1], ts[..., 2]

    def reset(self, seed=0):
        """Fresh worlds drawn on the device from combat.py:84-86."""
        self.engine.sample_reset(seed)
        return self.obs

    def load_state(self, pos, angle, vel=None):
        torch = _torch()
        t = self.engine.t
        E, N = self.engine.E, self.engine.N
        t["posvel"][..., 0:2] = torch.as_tensor(pos, dtype=torch.float32).reshape(E, N, 2).to(self.device)
        t["posvel"][..., 2:4] = 0 if vel is None else torch.as_tensor(vel, dtype=torch.float32).reshape(E, N, 2).to(self.device)
        t["angsleep"][..., 0] = torch.as_tensor(angle, dtype=torch.float32).reshape(E, N).to(self.device)
        self.engine.reset()
        return self.obs

    @property
    def obs(self):
        o = self.engine.t["obs"].view(self.engine.E, self.engine.N, self.engine.N, 4)
        return {"myHealth": self.health, "myTeam": self.engine.t["team"], "alive": self.alive,
                "agents": {"type": o[..., 3], "position": o[..., 0:3]}}

    @property
    def final_obs(self):
        """The terminal observation of each env's last finished match (keep_final=True), laid out as `obs`, with
        myHealth / alive from the final TDM state (valid rows: see final_info)."""
        f = self._final()
        o = f["obs"].view(self.engine.E, self.engine.N, self.engine.N, 4)
        ts = f["tdm_state"]
        return {"myHealth": ts[..., 0], "myTeam": self.engine.t["team"], "alive": (ts[..., 3].view(_torch().int32) & 1).bool(),
                "agents": {"type": o[..., 3], "position": o[..., 0:3]}}

    @property
    def rewards(self):
        return self.engine.t["rewards"]

    def step(self, actions):
        torch = _torch()
        E, N = self.engine.E, self.engine.N
        a = actions
        if not (torch.is_tensor(a) and a.dtype == torch.uint8 and a.is_cuda and tuple(a.shape) == (E, N, 4)
                and a.is_contiguous()):
            if self._act4 is None:
                self._act4 = torch.zeros((E, N, 4), dtype=torch.uint8, device=self.device)
            src = torch.as_tensor(actions, device=self.device)
            if src.dtype.is_floating_point or src.dtype == torch.bool:
                src = src.to(torch.uint8)
            a = self.engine.pack_actions(src.reshape(E, N, 4), self._act4)
        self.engine.step(a)
        self._check_overflow()
        return self.obs, self.engine.t["rewards"]

    def bot_actions(self, policy="random", seed=0, out=None):
        torch = _torch()
        if out is None:
            out = torch.empty((self.engine.E, self.engine.N, 4), dtype=torch.uint8, device=self.device)
        self.engine.bot_actions(_lib.BOTS[policy], seed, out)
        return out

    contacts = BatchedFlock.contacts
    rollout = BatchedFlock.rollout

    def close(self):
        self.engine.close()
