"""ctypes face of the CPU oracle (oracle/macm_oracle.c).

TEST INFRASTRUCTURE ONLY -- see the header of macm_oracle.c.  Only tests/,
``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline / ``--impl reference`` legs import
this module; nothing under ``gym-macm_b200/`` does.  PARITY UNPINNED (pybox2d not importable).
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libmacm_oracle.so")

FLOCK, TDM = 0, 1


class OParams(C.Structure):
    _fields_ = [
        ("env_kind", C.c_int), ("n_agents", C.c_int), ("n_targets", C.c_int),
        ("hz", C.c_double),
        ("velocity_iterations", C.c_int), ("position_iterations", C.c_int),
        ("radius", C.c_double), ("density", C.c_double), ("friction", C.c_double), ("linear_damping", C.c_double),
        ("agent_force", C.c_double), ("agent_rotation_speed", C.c_double),
        ("time_limit", C.c_double),
        ("reward_mode", C.c_int), ("action_mode", C.c_int), ("coord", C.c_int),
        ("reward_radius", C.c_double),
        ("damping_model", C.c_int), ("warm_starting", C.c_int), ("flags", C.c_int),
        ("cooldown_atk", C.c_double), ("cooldown_mov_penalty", C.c_double), ("melee_range", C.c_double),
        ("melee_dmg", C.c_double), ("percent_mov_penalty", C.c_double), ("init_health", C.c_double),
    ]


def build(force=False):
    """Compile the oracle with the committed recipe (oracle/Makefile)."""
    src = os.path.join(_HERE, "macm_oracle.c")
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-s", "-B"], env={**os.environ, "CC": "gcc"})
    return _LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            build()
        L = C.CDLL(_LIB_PATH)
        vp = C.c_void_p
        L.oracle_create.restype = vp
        L.oracle_create.argtypes = [C.POINTER(OParams), C.c_int]
        L.oracle_destroy.argtypes = [vp]
        L.oracle_reset.argtypes = [vp, vp, vp, vp, vp, vp]
        L.oracle_reset_env.argtypes = [vp, C.c_int, vp, vp, vp]
        L.oracle_flock_step.argtypes = [vp] * 9 + [C.c_int]
        L.oracle_flock_observe.argtypes = [vp] * 4
        L.oracle_tdm_step.argtypes = [vp] * 8 + [C.c_int]
        L.oracle_tdm_observe.argtypes = [vp] * 3
        L.oracle_get_bodies.argtypes = [vp, vp]
        L.oracle_get_contacts.restype = C.c_int
        L.oracle_get_contacts.argtypes = [vp, C.c_int, vp, vp, vp, C.c_int]
        L.oracle_set_env_state.argtypes = [vp, C.c_int, vp, C.c_int, vp, vp, vp, C.c_float, C.c_int, C.c_double, C.c_int]
        L.oracle_set_targets.argtypes = [vp, C.c_int, vp]
        L.oracle_get_tdm.argtypes = [vp, vp]
        L.oracle_get_env_info.argtypes = [vp, C.c_int, vp]
        L.oracle_world_create.restype = vp
        L.oracle_world_create.argtypes = [C.c_double] * 4 + [C.c_int]
        L.oracle_world_add_body.restype = C.c_int
        L.oracle_world_add_body.argtypes = [vp, C.c_double, C.c_double, C.c_double]
        L.oracle_world_set_angle.argtypes = [vp, C.c_int, C.c_double]
        L.oracle_world_get_angle.restype = C.c_double
        L.oracle_world_get_angle.argtypes = [vp, C.c_int]
        L.oracle_world_apply_force.argtypes = [vp, C.c_int, C.c_double, C.c_double]
        L.oracle_world_set_active.argtypes = [vp, C.c_int, C.c_int]
        L.oracle_world_set_warm_starting.argtypes = [vp, C.c_int]
        L.oracle_world_step.argtypes = [vp, C.c_double, C.c_int, C.c_int]
        L.oracle_world_raycast.restype = C.c_int
        L.oracle_world_raycast.argtypes = [vp, C.c_double, C.c_double, C.c_double, C.c_double, vp]
        _lib = L
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def default_params(env_kind=FLOCK, n_agents=4, n_targets=1, **kw):
    """settings.py:25-36 (fwSettings), :110-146 (flockSettings), :149-175 (combatSettings);
    combat.py:20-24 (Agent constants)."""
    p = dict(
        env_kind=env_kind, n_agents=n_agents, n_targets=n_targets, hz=60.0,
        velocity_iterations=8, position_iterations=3,
        radius=0.5, density=1.0, friction=0.3, linear_damping=5.0,
        agent_force=20.0, agent_rotation_speed=0.8 * (2 * np.pi), time_limit=60.0,
        reward_mode=0, action_mode=0, coord=0, reward_radius=7.0,
        damping_model=1, warm_starting=1, flags=1,
        cooldown_atk=1.0, cooldown_mov_penalty=0.5, melee_range=2.0, melee_dmg=0.25,
        percent_mov_penalty=0.2, init_health=1.0,
    )
    for k, v in kw.items():
        if k not in p:
            raise KeyError(k)
        p[k] = v
    if "reward_radius" not in kw:
        p["reward_radius"] = 7.0 if p["reward_mode"] == 0 else 1.0  # settings.py:146
    return p


class OracleBatch:
    """E independent worlds stepped by the scalar C oracle."""

    def __init__(self, n_envs, **params):
        self.params = default_params(**params)
        self.E = int(n_envs)
        self.N = int(self.params["n_agents"])
        self.T = int(self.params["n_targets"])
        self.kind = int(self.params["env_kind"])
        cp = OParams(**self.params)
        self._h = lib().oracle_create(C.byref(cp), self.E)
        if not self._h:
            raise ValueError("oracle_create rejected the parameters")
        self.target_idx = np.zeros(self.N, np.uint8)
        self.team = np.zeros(self.N, np.uint8)

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h and _lib is not None:
            _lib.oracle_destroy(h)

    # -- state ---------------------------------------------------------------------------------
    def reset(self, pos, angle, targets=None, target_idx=None, team=None):
        pos = np.ascontiguousarray(pos, np.float64).reshape(self.E, self.N, 2)
        angle = np.ascontiguousarray(angle, np.float64).reshape(self.E, self.N)
        if targets is not None:
            targets = np.ascontiguousarray(targets, np.float64).reshape(self.E, self.T, 2)
        if target_idx is not None:
            self.target_idx = np.ascontiguousarray(target_idx, np.uint8).reshape(self.N)
        if team is not None:
            self.team = np.ascontiguousarray(team, np.uint8).reshape(self.N)
        lib().oracle_reset(self._h, _p(pos), _p(angle), _p(targets), _p(self.target_idx), _p(self.team))

    def reset_env(self, ei, pos, angle, targets=None):
        """A new episode for env `ei` alone (fresh world, new bodies; target indices and teams are kept)."""
        pos = np.ascontiguousarray(pos, np.float64).reshape(self.N, 2)
        angle = np.ascontiguousarray(angle, np.float64).reshape(self.N)
        if targets is not None:
            targets = np.ascontiguousarray(targets, np.float64).reshape(self.T, 2)
        lib().oracle_reset_env(self._h, int(ei), _p(pos), _p(angle), _p(targets))

    def bodies(self):
        out = np.zeros((self.E, self.N, 10), np.float32)
        lib().oracle_get_bodies(self._h, _p(out))
        return out

    def contacts(self, ei):
        cap = self.N * (self.N - 1) // 2 + 1
        ab = np.zeros((cap, 2), np.int32)
        fl = np.zeros(cap, np.uint8)
        imp = np.zeros((cap, 2), np.float32)
        n = lib().oracle_get_contacts(self._h, ei, _p(ab), _p(fl), _p(imp), cap)
        return ab[:n].copy(), fl[:n].copy(), imp[:n].copy()

    def set_env_state(self, ei, body, ab, flags, imp, inv_dt0, step_count=0, time_passed=0.0, new_fixture=0):
        body = np.ascontiguousarray(body, np.float32).reshape(self.N, 10)
        ab = np.ascontiguousarray(ab, np.int32).reshape(-1, 2)
        flags = np.ascontiguousarray(flags, np.uint8)
        imp = np.ascontiguousarray(imp, np.float32).reshape(-1, 2)
        lib().oracle_set_env_state(self._h, ei, _p(body), len(ab), _p(ab), _p(flags), _p(imp), float(inv_dt0),
                                   int(step_count), float(time_passed), int(new_fixture))

    def set_targets(self, ei, targets):
        t = np.ascontiguousarray(targets, np.float32).reshape(self.T, 2)
        lib().oracle_set_targets(self._h, ei, _p(t))

    def env_info(self, ei):
        """touching: touching contacts after the last step's Collide; contacts: contacts at its end; peak_contacts:
        the most the world held at once during it (a fresh world's prologue can list pairs Collide then destroys)."""
        out = np.zeros(7, np.float64)
        lib().oracle_get_env_info(self._h, ei, _p(out))
        return dict(time_passed=out[0], done=int(out[1]), step_count=int(out[2]), inv_dt0=np.float32(out[3]),
                    touching=int(out[4]), contacts=int(out[5]), peak_contacts=int(out[6]))

    def tdm_state(self):
        out = np.zeros((self.E, self.N, 4), np.float64)
        lib().oracle_get_tdm(self._h, _p(out))
        return out

    # -- stepping ------------------------------------------------------------------------------
    def _flock_out(self):
        E, N = self.E, self.N
        return dict(nn_idx=np.zeros((E, N), np.int32), nn_pos=np.zeros((E, N, 3), np.float64),
                    tg_pos=np.zeros((E, N, 3), np.float64), rewards=np.zeros((E, N), np.float64),
                    collided=np.zeros((E, N), np.uint8), done=np.zeros(E, np.uint8))

    def flock_step(self, actions, n_threads=1):
        o = self._flock_out()
        if self.params["action_mode"] == 0:
            a = np.ascontiguousarray(actions, np.int32).reshape(self.E, self.N, 3)
            ad, ac = _p(a), None
        else:
            a = np.ascontiguousarray(actions, np.float64).reshape(self.E, self.N, 2)
            ad, ac = None, _p(a)
        lib().oracle_flock_step(self._h, ad, ac, _p(o["nn_idx"]), _p(o["nn_pos"]), _p(o["tg_pos"]), _p(o["rewards"]),
                                _p(o["collided"]), _p(o["done"]), int(n_threads))
        return o

    def flock_observe(self):
        o = self._flock_out()
        lib().oracle_flock_observe(self._h, _p(o["nn_idx"]), _p(o["nn_pos"]), _p(o["tg_pos"]))
        return {k: o[k] for k in ("nn_idx", "nn_pos", "tg_pos")}

    def _tdm_out(self):
        E, N = self.E, self.N
        return dict(obs=np.zeros((E, N, N, 3), np.float64), type=np.zeros((E, N, N), np.int8),
                    rewards=np.zeros((E, N), np.float64), collided=np.zeros((E, N), np.uint8),
                    done=np.zeros(E, np.uint8), winner=np.zeros(E, np.int32))

    def tdm_step(self, actions, n_threads=1):
        o = self._tdm_out()
        a = np.ascontiguousarray(actions, np.int32).reshape(self.E, self.N, 4)
        lib().oracle_tdm_step(self._h, _p(a), _p(o["obs"]), _p(o["type"]), _p(o["rewards"]), _p(o["collided"]),
                              _p(o["done"]), _p(o["winner"]), int(n_threads))
        return o

    def tdm_observe(self):
        o = self._tdm_out()
        lib().oracle_tdm_observe(self._h, _p(o["obs"]), _p(o["type"]))
        return {k: o[k] for k in ("obs", "type")}


class OracleWorld:
    """One world driven body by body, the way the reference drives pybox2d."""

    def __init__(self, radius=0.5, density=1.0, friction=0.3, linear_damping=5.0, damping_model=1):
        self._h = lib().oracle_world_create(radius, density, friction, linear_damping, damping_model)
        self.n = 0

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h and _lib is not None:
            _lib.oracle_destroy(h)

    def add_body(self, x, y, angle):
        i = lib().oracle_world_add_body(self._h, float(x), float(y), float(angle))
        if i < 0:
            raise RuntimeError("oracle world is full")
        self.n = i + 1
        return i

    def set_angle(self, i, a):
        lib().oracle_world_set_angle(self._h, i, float(a))

    def get_angle(self, i):
        return lib().oracle_world_get_angle(self._h, i)

    def apply_force(self, i, fx, fy):
        lib().oracle_world_apply_force(self._h, i, float(fx), float(fy))

    def set_active(self, i, flag):
        lib().oracle_world_set_active(self._h, i, int(bool(flag)))

    def set_warm_starting(self, flag):
        lib().oracle_world_set_warm_starting(self._h, int(bool(flag)))

    def step(self, dt, vel_iters, pos_iters):
        lib().oracle_world_step(self._h, float(dt), int(vel_iters), int(pos_iters))

    def raycast(self, p1, p2):
        fr = C.c_double(1.0)
        hit = lib().oracle_world_raycast(self._h, float(p1[0]), float(p1[1]), float(p2[0]), float(p2[1]), C.byref(fr))
        return hit, fr.value

    def bodies(self):
        out = np.zeros((1, max(self.n, 1), 10), np.float32)
        lib().oracle_get_bodies(self._h, _p(out))
        return out[0, : self.n]

    def contacts(self):
        cap = max(self.n * (self.n - 1) // 2, 1)
        ab = np.zeros((cap, 2), np.int32)
        fl = np.zeros(cap, np.uint8)
        imp = np.zeros((cap, 2), np.float32)
        n = lib().oracle_get_contacts(self._h, 0, _p(ab), _p(fl), _p(imp), cap)
        return ab[:n].copy(), fl[:n].copy(), imp[:n].copy()
