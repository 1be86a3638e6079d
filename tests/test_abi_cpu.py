"""CPU-side checks: libmacm.so loads and exports every symbol include/macm.h declares, the ctypes
structs match the header, and the host marshalling helpers do what the reference's dict API does.
No compute call is made (there is no GPU here)."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as g
    g.build()
    from gym_macm import _lib
    return _lib


def test_every_declared_symbol_is_exported(built):
    hdr = open(os.path.join(ROOT, "include", "macm.h")).read()
    declared = set(re.findall(r"\b(macm_[a-z_0-9]+)\s*\(", hdr))
    assert declared, "no declarations found"
    L = built.lib()
    for name in sorted(declared):
        assert hasattr(L, name), "libmacm.so does not export %s" % name
    assert declared == set(built.EXPORTS)


def test_struct_layout_matches_header(built):
    # field order of the ctypes mirrors == member order of the C structs
    hdr = open(os.path.join(ROOT, "include", "macm.h")).read()
    body = hdr[hdr.index("typedef struct macm_params {"):hdr.index("} macm_params;")]
    names = []
    for line in body.splitlines()[1:]:
        line = line.split("/*")[0].strip()
        m = re.match(r"(int32_t|double)\s+([^;]+);", line)
        if m:
            names += [n.strip() for n in m.group(2).split(",")]
    assert names == [f[0] for f in built.MacmParams._fields_]
    body = hdr[hdr.index("typedef struct macm_buffers {"):hdr.index("} macm_buffers;")]
    names = re.findall(r"^\s*(?:float|uint32_t|int32_t|uint8_t)\*\s+(\w+);", body, re.M)
    assert tuple(names) == built.BUFFER_NAMES
    body = hdr[hdr.index("typedef struct macm_rollout_out {"):hdr.index("} macm_rollout_out;")]
    names = re.findall(r"^\s*(?:float|int32_t|uint8_t)\*\s+(\w+);", body, re.M)
    assert names == [f[0] for f in built.MacmRolloutOut._fields_]


def test_defaults_are_the_reference_settings(built):
    p = built.default_params(built.FLOCK)
    assert (p.hz, p.velocity_iterations, p.position_iterations, p.warm_starting) == (60.0, 8, 3, 1)
    assert (p.radius, p.density, p.friction, p.linear_damping) == (0.5, 1.0, 0.3, 5.0)
    assert p.agent_force == 20.0 and p.agent_rotation_speed == 0.8 * (2 * np.pi) and p.time_limit == 60.0
    assert p.reward_radius == 7.0 and (p.target_mindist, p.target_maxdist, p.start_spread) == (25.0, 60.0, 20.0)
    t = built.default_params(built.TDM)
    assert (t.cooldown_atk, t.cooldown_mov_penalty, t.melee_range, t.melee_dmg) == (1.0, 0.5, 2.0, 0.25)


_NO_DEVICE = r"""
import ctypes as C
import pytest
import gym_macm
from gym_macm import _lib as built
with pytest.raises(built.MacmError):
    gym_macm.BatchedFlock(4, n_agents=[4])
with pytest.raises(built.MacmError):
    gym_macm.make("gym_macm:cm-flock-v0", n_agents=[4])
# macm_create itself refuses without a device
p = built.default_params(built.FLOCK)
h = C.c_void_p()
assert built.lib().macm_create(C.byref(h), C.byref(p), 0) == -2 and not h
p.n_agents = 129      # MACM_MAX_AGENTS is 128
assert built.lib().macm_create(C.byref(h), C.byref(p), 0) == -1
"""


def test_no_cpu_fallback(built):
    # in a child process that sees no CUDA device, so that the check also runs where a GPU is present
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="",
               PYTHONPATH=os.pathsep.join([ROOT, os.path.join(ROOT, "gym-macm_b200")]))
    r = subprocess.run([sys.executable, "-c", _NO_DEVICE], capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode == 0, r.stderr


def test_settings_bag():
    from gym_macm.settings import flockSettings
    s = flockSettings()
    assert s.hz == 60.0 and s.velocityIterations == 8 and s.positionIterations == 3
    assert s.reward_mode == "binary" and s.reward_radius == 7 and s.coord == "polar"
    assert s.bodySettings["linearDamping"] == 5 and s.bodySettings["fixedRotation"] is True
    s = flockSettings(reward_mode="linear", time_limit=10, hz=30.0)
    assert s.reward_radius == 1 and s.time_limit == 10 and s.hz == 30.0  # settings.py:143-146


def test_dict_marshalling():
    from gym_macm.envs.mvmnt import encode_discrete_actions, obs_to_dict, rewards_to_dict
    ids = [0, 1, 2]
    a = encode_discrete_actions({0: np.array([2, 1, 0]), 1: [1, 1, 1], 2: (0, 2, 2)}, ids)
    assert a.dtype == np.uint8 and a.tolist() == [[2, 1, 0, 0], [1, 1, 1, 0], [0, 2, 2, 0]]
    obs = np.arange(12, dtype=np.float32).reshape(3, 4)
    d = obs_to_dict(ids, np.array([1, 0, 1]), obs, 3)
    assert set(d) == {0, 1, 2} and [n["type"] for n in d[0]["nodes"]] == [0, 1]
    assert d[0]["nodes"][0]["id"] == 1 and d[0]["nodes"][1]["id"] == 3
    assert d[2]["nodes"][0]["position"].dtype == np.float64 and d[2]["nodes"][0]["position"].tolist() == [8.0, 9.0]
    assert d[2]["nodes"][1]["position"].tolist() == [10.0, 11.0]
    r = rewards_to_dict(ids, np.array([1.0, 0.0, -1.0], np.float32), np.array([0, 0, 1]), "binary")
    assert r == {0: 1, 1: 0, 2: -1} and all(isinstance(v, int) for v in r.values())
    r = rewards_to_dict(ids, np.array([0.25, 0.5, -1.0], np.float32), np.array([0, 0, 1]), "linear")
    assert r[0] == 0.25 and isinstance(r[0], np.float64) and r[2] == -1


def test_spaces_contains():
    from gym_macm import spaces
    sp = spaces.Dict({0: spaces.MultiDiscrete([3, 3, 3]), 1: spaces.MultiDiscrete([3, 3, 3])})
    assert sp.contains({0: np.array([0, 1, 2]), 1: np.array([2, 2, 2])})
    assert not sp.contains({0: np.array([0, 1, 3]), 1: np.array([2, 2, 2])})
    assert not sp.contains({0: np.array([0, 1, 2])})


def test_host_bots_match_reference_rules():
    from gym_macm import bots
    obs = {3: {"nodes": [{"type": 0, "id": 1, "position": np.array([2.0, 0.1])},
                         {"type": 1, "id": 4, "position": np.array([10.0, 0.5])}]}}
    assert bots.flock(obs).tolist() == [2, 1, 2]      # |0.5| < pi/4 -> forward; sign(+) + 1 = 2
    obs[3]["nodes"][1]["position"] = np.array([10.0, -2.0])
    assert bots.flock(obs).tolist() == [1, 1, 0]
    obs[3]["nodes"][1]["position"] = np.array([0.5, -2.0])
    assert bots.flock(obs).tolist() == [1, 1, 1]      # inside 1 m: idle
