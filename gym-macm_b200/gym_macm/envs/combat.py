"""`TDM`: team deathmatch, dict-in/dict-out, one world = a batch of one on the CUDA simulator.

The reference class (gym_macm/envs/combat.py:56-264) cannot be constructed as shipped
(`combatSettings` is never imported, SURVEY.md Appendix B8); this host keeps its interface --
`TDM(render, n_agents=[..per team..], actors, colors, **kwargs)`, string agent ids
`str(team) + str(j)` (combat.py:87), `obs[id] = {"myHealth", "myTeam", "agents": [...]}`
(combat.py:211-226), `done`, `winner`, `n_alive` -- with the repaired semantics the batched
kernel and the oracle implement, and returns `(obs, rewards)` from `step` (Appendix B12).
"""
import random

import numpy as np

from gym_macm import spaces
from gym_macm.batched import BatchedTDM, _as_list
from gym_macm.envs.mvmnt import check_capacity

try:  # pragma: no cover
    import gym as _gym
    _Base = _gym.Env
except Exception:
    try:  # pragma: no cover
        import gymnasium as _gym
        _Base = _gym.Env
    except Exception:
        _Base = object


class Agent(object):
    """combat.Agent (combat.py:13-54): constants plus live values read back from the device."""

    def __init__(self, env, index, ID, team=0, actor=None):
        self._env, self._i = env, index
        self.init_health = env.settings.init_health
        self.team = team
        self.id = ID
        self.actor = actor
        self.rotation_speed = env.settings.agent_rotation_speed
        self._force = env.settings.agent_force
        self.melee_range = env.settings.melee_range
        self.melee_dmg = env.settings.melee_dmg
        self.percent_mov_penalty = env.settings.percent_mov_penalty

    @property
    def health(self):
        return float(self._env._tdm()[0][self._i])

    @property
    def alive(self):
        return bool(self._env._tdm()[3][self._i])

    @property
    def cooldown_atk(self):
        return self._env._tdm()[1][self._i] / self._env.settings.hz

    @property
    def cooldown_mov_penalty(self):
        return self._env._tdm()[2][self._i] / self._env.settings.hz

    @property
    def force(self):
        return self._force * (1 - self.percent_mov_penalty * int(self.cooldown_mov_penalty > 0))


def tdm_obs_to_dict(ids, teams, health, alive, obs):
    """Arrays -> the reference's obs dict (combat.py:206-227): alive agents only, others in index order."""
    out = {}
    for i, aid in enumerate(ids):
        if not alive[i]:
            continue
        others = [{"type": int(obs[i, j, 3]), "position": np.array(obs[i, j, 0:3], dtype=np.float64)}
                  for j in range(len(ids)) if obs[i, j, 3] >= 0]
        out[aid] = {"myHealth": np.array([health[i]], dtype=np.float64), "myTeam": teams[i], "agents": others}
    return out


def encode_tdm_actions(actions, ids, alive):
    out = np.ones((len(ids), 4), np.uint8)
    out[:, 3] = 0
    for k, i in enumerate(ids):
        if alive[k]:
            out[k] = np.asarray(actions[i]).reshape(-1)[:4]
    return out


class TDM(_Base):
    name = "Team Deathmatch"
    description = ("TDM on an empty world")

    def __init__(self, render="False", n_agents=[1, 1], actors=None, colors=None, device=None, **kwargs):
        if render is True:
            raise NotImplementedError("rendering stays with the reference's CPU backends")
        if kwargs.get("obs_dtype", "float32") != "float32":
            # the reference's dicts hold Python floats of the fp32 observation; a rounded one would not be it
            raise ValueError("%s returns the reference's float observations: obs_dtype must be float32 "
                             "(16-bit observations are for the batched classes)" % type(self).__name__)
        n_agents = _as_list(n_agents)
        nn = sum(n_agents)
        kwargs.setdefault("max_contacts", max(1, nn * (nn - 1) // 2))   # one world: full capacity (see mvmnt.Flock)
        kwargs.setdefault("max_touching", max(1, nn * (nn - 1) // 2))   # beyond 240: the global-memory solver stage
        self._batch = BatchedTDM(1, n_agents=n_agents, device=device, seed=None, **kwargs)
        self.settings = self._batch.settings
        self.done = False
        self.winner = None
        self.n_agents = n_agents
        self.world_width = self.settings.world_width
        self.world_height = self.settings.world_height
        self.time_passed = 0
        self.agents = []
        N = sum(n_agents)
        pos, ang = np.zeros((N, 2)), np.zeros(N)
        k = 0
        for i in range(len(n_agents)):   # same draws, same order as combat.py:82-86
            for j in range(n_agents[i]):
                pos[k, 0] = random.random() * (i + self.world_width / 2)
                pos[k, 1] = random.random() * self.world_height
                ang[k] = random.uniform(-1, 1) * np.pi
                agent = Agent(self, k, ID=str(i) + str(j), team=i)
                if actors:
                    agent.actor = actors[i][j]
                if colors:
                    agent._color = colors[i]
                self.agents.append(agent)
                k += 1
        self._ids = [a.id for a in self.agents]
        self._teams = [a.team for a in self.agents]
        self._cache = None
        self._batch.load_state(pos[None], ang[None])
        self.n_alive = list(n_agents)
        self.create_space()
        self.create_space_flag = False
        self.obs = self.get_obs()

    def _tdm(self):
        if self._cache is None:
            ts = self._batch.state["tdm_state"][0].cpu()
            import torch
            ti = ts.view(torch.int32).numpy()
            self._cache = (ts[:, 0].numpy().copy(), ti[:, 1].copy(), ti[:, 2].copy(), (ti[:, 3] & 1).astype(bool))
        return self._cache

    def step(self, actions=None):
        if self.done:
            self.quit()
        alive = self._tdm()[3]
        if actions is None:
            actions = {}
            for agent in self.agents:
                if agent.alive:
                    actions[agent.id] = agent.actor(self.obs[agent.id])
        assert self.action_space.contains(actions)
        import torch
        a = torch.from_numpy(encode_tdm_actions(actions, self._ids, alive)[None])
        out = self._batch.engine.step_host(a, want=("rewards", "collided", "done"))
        self._cache = None
        check_capacity(self._batch)
        rewards = {aid: (-1 if out["rewards"][0, k] < 0 else 0) for k, aid in enumerate(self._ids)
                   if self._tdm()[3][k]}
        self.obs = self.get_obs(observe=False)
        self.time_passed += (1 / self.settings.hz)
        alive = self._tdm()[3]
        self.n_alive = [int(sum(alive[k] for k, t in enumerate(self._teams) if t == team))
                        for team in range(len(self.n_agents))]
        alive_teams = [i for i, e in enumerate(self.n_alive) if e != 0]
        if self.time_passed > self.settings.time_limit:
            self.done = True
        if len(alive_teams) == 1:
            self.done = True
            self.winner = alive_teams[0]
        if len(alive_teams) == 0:
            self.done = True
        self.create_space()
        return self.obs, rewards

    def create_space(self):
        alive = [a for a in self.agents if a.alive]
        self.action_space = spaces.Dict({a.id: spaces.MultiDiscrete([3, 3, 3, 2]) for a in alive})
        other = spaces.Dict({"type": spaces.Discrete(1),
                             "position": spaces.Box(np.array([0, -np.pi, -np.pi]), np.array([np.inf, np.pi, np.pi]))})
        self.observation_space = spaces.Dict(
            {a.id: spaces.Dict({"myHealth": spaces.Box(low=0, high=1, shape=(1,)), "myTeam": spaces.Discrete(1),
                                "agents": spaces.Tuple([other] * (len(alive) - 1))}) for a in alive})

    def get_rewards(self):
        t = self._batch.state
        r = t["rewards"][0].cpu().numpy()
        return {aid: (-1 if r[k] < 0 else 0) for k, aid in enumerate(self._ids) if self._tdm()[3][k]}

    def get_obs(self, observe=True):
        if observe:
            self._batch.engine.observe()
        t = self._batch.state
        N = len(self.agents)
        h, _, _, alive = self._tdm()
        return tdm_obs_to_dict(self._ids, self._teams, h, alive, t["obs"][0].cpu().numpy().reshape(N, N, 4))

    def reset(self):
        """Repaired (App. B13): new positions, full health, everyone alive again."""
        self.done, self.winner, self.time_passed = False, None, 0
        N = len(self.agents)
        pos, ang = np.zeros((N, 2)), np.zeros(N)
        for k, agent in enumerate(self.agents):
            pos[k, 0] = random.random() * (agent.team + self.world_width / 2)
            pos[k, 1] = random.random() * self.world_height
            ang[k] = random.uniform(-1, 1) * np.pi
        self._cache = None
        self._batch.load_state(pos[None], ang[None])
        self.n_alive = list(self.n_agents)
        self.create_space()
        self.obs = self.get_obs()
        return self.obs

    def BeginContact(self, agent1, agent2):
        pass

    def CheckKeys(self, *args):
        pass

    def render(self, mode="rgb_array", size=(480, 640), view=None):
        """This env as a top-down RGB picture drawn on the device: numpy uint8 [H,W,3] (size = (H, W)), row 0 at the
        top.  view = (centre x, centre y, half-width in metres), or None to fit every agent.  Only mode
        "rgb_array": the reference's pyglet window stays with its CPU backends."""
        if mode != "rgb_array":
            raise NotImplementedError("only render(mode=\"rgb_array\") is drawn here; the reference's pyglet window "
                                      "stays with its CPU backends")
        return self._batch.render(size, views=None if view is None else [view])[0].cpu().numpy()

    def render_state(self):
        """The objects the reference's CPU renderer reads (pyglet_framework.py:122-180), see gym_macm.render."""
        return self._batch.render_state(0)

    def quit(self):
        return

    def close(self):
        self._batch.close()
