"""Settings bags with the reference's attribute names (gym_macm/settings.py:25-59,110-175).

Same defaults, same `**kwargs` override rule (settings.py:143-144), same derived
`reward_radius` (settings.py:146).  `combatSettings` accepts kwargs too (the reference's ignores
them, SURVEY App. B8) and carries the Agent constants of combat.py:20-24.  Box2D objects are
replaced by plain records: the circle fixture is data for the CUDA engine, not a b2FixtureDef.
"""
import numpy as np


class CircleFixture(object):
    """Stands in for b2FixtureDef(shape=b2CircleShape(radius), density, friction) (settings.py:127-132)."""

    def __init__(self, radius=0.5, density=1, friction=0.3):
        self.radius, self.density, self.friction = radius, density, friction

    def __repr__(self):
        return "CircleFixture(radius=%r, density=%r, friction=%r)" % (self.radius, self.density, self.friction)


class fwSettings(object):
    backend = 'no_render'
    # physics options (settings.py:29-36)
    hz = 60.0
    velocityIterations = 8
    positionIterations = 3
    enableWarmStarting = True
    enableContinuous = True   # every agent is a non-bullet dynamic body: SolveTOI skips all contacts
    enableSubStepping = False
    # drawing flags kept so host code that reads them keeps working; rendering is off the hot path
    drawStats = False
    drawShapes = True
    drawJoints = True
    drawCoreShapes = False
    drawAABBs = False
    drawOBBs = False
    drawPairs = False
    drawContactPoints = False
    maxContactPoints = 100
    drawContactNormals = False
    drawFPS = False
    drawMenu = True
    drawCOMs = False
    pointSize = 2.5
    pause = False
    singleStep = False
    onlyInit = False


class _EnvSettings(fwSettings):
    def _common(self):
        self.render = False
        self.record = False
        self.record_dir = "../imgs/"
        self.verbose_display = True
        self.start_spread = 20
        self.start_point = [0, 0]
        self.agent_rotation_speed = 0.8 * (2 * np.pi)
        self.agent_force = 20
        self.time_limit = 60
        self.bodySettings = {"fixtures": CircleFixture(0.5, 1, 0.3), "linearDamping": 5, "fixedRotation": True}
        # engine knobs the reference cannot express (pybox2d's Box2D version is unpinned)
        # Box2D changed its damping formula between 2.3.0 and 2.3.1 (0.7 % per step at the reference's settings).
        # The reference calls ApplyForce(..., wake=) and installs pybox2d from pip, whose releases (Box2D 2.3.2+,
        # box2d-py 2.3.5+) bundle the later engine: "pade" is the default.  tests/test_pybox2d_probe.py checks this
        # against the real engine the day one is importable.
        self.damping_model = "pade"        # "pade": v *= 1/(1 + h c), Box2D >= 2.3.1; "taylor": v *= clamp(1 - h c, 0, 1), <= 2.3.0
        self.max_contacts = 0              # 0 = library default
        self.max_touching = 0
        self.env_index_base = 0            # global index of this batch's env 0 (gym_macm.dist shards)
        # batched hosts only (the reference has one world and a broken reset(), SURVEY App. B3):
        self.auto_reset = False            # an env whose `done` flag is set starts a new episode right after the step
        self.keep_final = False            # keep each reset env's terminal observation and outcome (final_obs, final_info)
        self.check_overflow = False        # debug: step() raises when an env ran out of contact capacity
        # element type of every observation: "float32", or "float16" / "bfloat16" -- the fp32 value rounded once to
        # nearest even on the device, half the bytes through HBM, PCIe and NVLink; the simulation does not change
        self.obs_dtype = "float32"


class flockSettings(_EnvSettings):
    def __init__(self, **kwargs):
        super(flockSettings, self).__init__()
        self._common()
        # task (settings.py:135-141)
        self.action_mode = "discrete"
        self.reward_mode = "binary"
        self._reward_radius = 7
        self.target_mindist = 25
        self.target_maxdist = 60
        self.coord = "polar"
        for kw in kwargs:
            setattr(self, kw, kwargs[kw])
        self.reward_radius = self._reward_radius if self.reward_mode == "binary" else 1


class combatSettings(_EnvSettings):
    def __init__(self, **kwargs):
        super(combatSettings, self).__init__()
        self._common()
        self.cooldown_atk = 1             # settings.py:165
        self.cooldown_mov_penalty = 0.5   # settings.py:166
        # combat.Agent constants (combat.py:15,20-24)
        self.init_health = 1
        self.melee_range = 2
        self.melee_dmg = 0.25
        self.percent_mov_penalty = 0.2
        self.world_width = 30             # combat.py:76-77
        self.world_height = 30
        self.repair_mov_cooldown = True   # SURVEY App. B10
        self.coord = "polar"
        self.action_mode = "discrete"
        for kw in kwargs:
            setattr(self, kw, kwargs[kw])
