"""`Flock`: the single-environment, dict-in/dict-out face of the batched CUDA simulator.

Drop-in for the reference class of the same name (gym_macm/envs/mvmnt.py:27-272): same
constructor, same attributes (`obs`, `agents`, `done`, `targets`, `settings`, `action_space`,
`observation_space`, `time_passed`), same `step(actions=None) -> (obs, rewards)` 2-tuple, same
obs/reward dict layout.  One world is simply a batch of one: every number comes from
libmacm.so through `BatchedFlock.step_host`; this file only converts between dicts and arrays.
"""
import random

import numpy as np

from gym_macm import spaces
from gym_macm.batched import BatchedFlock, _as_list

try:  # pragma: no cover
    import gym as _gym
    _Base = _gym.Env
except Exception:
    try:  # pragma: no cover
        import gymnasium as _gym
        _Base = _gym.Env
    except Exception:
        _Base = object


class Body(object):
    """Read-only view of one agent's rigid body (what host code reads from `agent.body`)."""

    def __init__(self, env, index):
        self._env, self._i = env, index

    @property
    def position(self):
        return self._env._state()[0][self._i, 0:2].astype(np.float64)

    @property
    def linearVelocity(self):
        return self._env._state()[0][self._i, 2:4].astype(np.float64)

    @property
    def angle(self):
        return float(self._env._state()[1][self._i, 0])


class Agent(object):
    def __init__(self, settings, ID, actor=None):
        self.id = ID
        self.actor = actor
        self.rotation_speed = settings.agent_rotation_speed
        self.force = settings.agent_force
        self._color = (0.4, 0.4, 0.6)
        self.color = (0.4, 0.4, 0.6)

    def reset_color(self):
        self.color = self._color


def check_capacity(batch):
    """The dict API never returns results that silently differ from the reference's: a world that ran out of
    contact capacity raises (cannot happen with the capacities the dict API asks for: every pair)."""
    from gym_macm._lib import ENV_CONTACT_OVERFLOW, ENV_TOUCH_OVERFLOW, MacmError
    if int(batch.state["env_state"][0, 1]) & (ENV_CONTACT_OVERFLOW | ENV_TOUCH_OVERFLOW):
        raise MacmError("the world holds more contacts than the simulator's capacity (max_contacts=%d, max_touching=%d)"
                        % (batch.engine.C, batch.engine.sizes.max_touching))


# ---- pure marshalling helpers (no device needed; covered by the CPU tests) --------------------
def encode_discrete_actions(actions, ids, width=3):
    """{id: [a0, a1, a2(, a3)]} -> uint8 [N, 4] in agent order."""
    out = np.zeros((len(ids), 4), np.uint8)
    for k, i in enumerate(ids):
        a = np.asarray(actions[i]).reshape(-1)
        out[k, :width] = a[:width]
    return out


def encode_continuous_actions(actions, ids):
    return np.asarray([np.asarray(actions[i], np.float64).reshape(2) for i in ids], np.float32)


def obs_to_dict(ids, nn_idx, obs, n_agents):
    """Arrays -> the reference's obs dict (mvmnt.py:186,204-220): two nodes per agent."""
    D = obs.shape[-1] // 2
    out = {}
    for k, i in enumerate(ids):
        out[i] = {"nodes": [
            {"type": 0, "id": ids[int(nn_idx[k])] if nn_idx[k] >= 0 else None,
             "position": np.array(obs[k, 0:D], dtype=np.float64)},
            {"type": 1, "id": n_agents, "position": np.array(obs[k, D:2 * D], dtype=np.float64)}]}
    return out


def rewards_to_dict(ids, rewards, collided, reward_mode):
    """-1 for agents in any contact, else int 0/1 (binary) or float (linear) (mvmnt.py:160-179)."""
    out = {}
    for k, i in enumerate(ids):
        if collided[k]:
            out[i] = -1
        elif reward_mode == "binary":
            out[i] = int(rewards[k])
        else:
            out[i] = np.float64(rewards[k])
    return out


class Flock(_Base):
    name = "Flock v0"
    description = ("Flock")

    def __init__(self, n_agents=[10], actors=None, colors=None, targets=None, device=None, **kwargs):
        if kwargs.get("obs_dtype", "float32") != "float32":
            # the reference's dicts hold Python floats of the fp32 observation; a rounded one would not be it
            raise ValueError("%s returns the reference's float observations: obs_dtype must be float32 "
                             "(16-bit observations are for the batched classes)" % type(self).__name__)
        n_agents = _as_list(n_agents)
        # one world: room for every possible pair in the contact list and in the solver's stage, so that no pile
        # can run out of contact capacity (a batch trades that for shared memory, see BatchedFlock.overflowed)
        nn = sum(n_agents)
        kwargs.setdefault("max_contacts", max(1, nn * (nn - 1) // 2))
        kwargs.setdefault("max_touching", max(1, nn * (nn - 1) // 2))   # beyond 240: the global-memory solver stage
        self._batch = BatchedFlock(1, n_agents=n_agents, actors=actors, colors=colors, targets=targets,
                                   device=device, seed=None, **kwargs)
        self.settings = self._batch.settings
        if self.settings.render:
            raise NotImplementedError("rendering stays with the reference's CPU backends; use render=False")
        self.done = False
        self.n_agents = n_agents
        self.n_targets = self._batch.n_targets
        self.targets_idx = self._batch.targets_idx
        self.time_passed = 0
        N = sum(n_agents)

        # same draws, in the same order, from the same global generator as mvmnt.py:48-52,62-64
        self.t_min, self.t_max = self.settings.target_mindist, self.settings.target_maxdist
        self.targets = []
        for t in range(self.n_targets):
            rand_angle = 2 * np.pi * random.random()
            rand_dist = self.t_min + random.random() * (self.t_max - self.t_min)
            self.targets.append(np.array([rand_dist * np.cos(rand_angle), rand_dist * np.sin(rand_angle)]))
        self.agents = []
        pos, ang = np.zeros((N, 2)), np.zeros(N)
        for i in range(N):
            pos[i, 0] = self.settings.start_spread * (random.random() - 0.5) + self.settings.start_point[0]
            pos[i, 1] = self.settings.start_spread * (random.random() - 0.5) + self.settings.start_point[1]
            ang[i] = random.uniform(-1, 1) * np.pi
            agent = Agent(self.settings, ID=i)
            if actors:
                agent.actor = actors[i]
            if colors:
                agent._color = colors[i]
            agent.body = Body(self, i)
            self.agents.append(agent)
        self._ids = [a.id for a in self.agents]
        self._cache = None
        self._batch.load_state(pos[None], ang[None], targets=np.asarray(self.targets)[None])
        self.create_space()
        self.create_space_flag = False
        self.obs = self.get_obs()

    # -- helpers -------------------------------------------------------------------------------
    def _state(self):
        if self._cache is None:
            t = self._batch.state
            self._cache = (t["posvel"][0].cpu().numpy(), t["angsleep"][0].cpu().numpy())
        return self._cache

    def _push_targets(self):
        import torch
        self._batch.targets.copy_(torch.as_tensor(np.asarray(self.targets, np.float32)[None]))

    # -- the reference's interface ------------------------------------------------------------------
    def step(self, actions=None):
        if self.done:
            self.quit()
        if actions is None:
            actions = {}
            for agent in self.agents:
                actions[agent.id] = agent.actor({agent.id: self.obs[agent.id]})
        assert self.action_space.contains(actions)

        import torch
        if self.settings.action_mode == "discrete":
            a = torch.from_numpy(encode_discrete_actions(actions, self._ids)[None])
        else:
            a = torch.from_numpy(encode_continuous_actions(actions, self._ids)[None])
        out = self._batch.engine.step_host(a)
        self._cache = None
        check_capacity(self._batch)
        rewards = rewards_to_dict(self._ids, out["rewards"][0].numpy(), out["collided"][0].numpy(),
                                  self.settings.reward_mode)
        self.time_passed += (1 / self.settings.hz)
        if self.time_passed > self.settings.time_limit:
            self.done = True
        self.obs = obs_to_dict(self._ids, out["nn_idx"][0].numpy(), out["obs"][0].numpy(), len(self.agents))
        return self.obs, rewards

    def create_space(self):
        if self.settings.action_mode == "discrete":
            self.action_space = spaces.Dict({agent.id: spaces.MultiDiscrete([3, 3, 3]) for agent in self.agents})
        if self.settings.action_mode == "continuous":
            self.action_space = spaces.Dict({agent.id: spaces.Box(np.array([-1, -1]), np.array([1, 1]))
                                             for agent in self.agents})
        node = spaces.Dict({"type": spaces.Discrete(1), "id": spaces.Discrete(1),
                            "position": spaces.Box(np.array([0, -np.pi]), np.array([np.inf, np.pi]))})
        self.observation_space = spaces.Dict(
            {agent.id: spaces.Dict({"nodes": spaces.Tuple([node] * (len(self.agents) + 1))}) for agent in self.agents})

    def get_rewards(self):
        t = self._batch.state
        return rewards_to_dict(self._ids, t["rewards"][0].cpu().numpy(), t["collided"][0].cpu().numpy(),
                               self.settings.reward_mode)

    def get_obs(self):
        self._batch.engine.observe()
        t = self._batch.state
        return obs_to_dict(self._ids, t["nn_idx"][0].cpu().numpy(), t["obs"][0].cpu().numpy(), len(self.agents))

    def reset(self):
        """Repaired (SURVEY App. B3): re-draw positions and angles as the reference intends
        (mvmnt.py:228-232) and also zero velocities, contacts and the clock."""
        self.done = False
        self.time_passed = 0
        N = len(self.agents)
        pos, ang = np.zeros((N, 2)), np.zeros(N)
        for i in range(N):
            pos[i, 0] = self.settings.start_spread * (random.random() - 0.5) + self.settings.start_point[0]
            pos[i, 1] = self.settings.start_spread * (random.random() - 0.5) + self.settings.start_point[1]
            ang[i] = random.uniform(-1, 1) * np.pi
        self._cache = None
        self._batch.load_state(pos[None], ang[None], targets=np.asarray(self.targets)[None])
        self.create_space()
        self.obs = self.get_obs()
        return self.obs

    def run(self):
        while not self.done:
            self.step()

    def MouseDown(self, p, selected_target=0):
        """Move a target (mvmnt.py:261-265)."""
        self.targets[selected_target] = np.asarray(p, np.float64)
        self._push_targets()

    def BeginContact(self, agent1, agent2):
        pass

    def render_state(self):
        """The objects the reference's CPU renderer reads (pyglet_framework.py:122-180), see gym_macm.render."""
        return self._batch.render_state(0)

    def quit(self):
        return

    def close(self):
        self._batch.close()
