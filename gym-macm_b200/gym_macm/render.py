"""Frames of the envs (SURVEY 8(f4)): the state export for the reference's CPU renderer, and the device frames.

Rendering stays in the reference (gym_macm/backends/pyglet_framework.py, off the hot path); what it needs from the
simulator is, per frame, the few attributes `PygletDraw.ManualDraw` reads (pyglet_framework.py:122-180,361-383):

    for body in test.world.bodies:  body.transform.position / .angle, body.userData.color (.r .g .b, `color / 3`
                                    for an inactive body), body.active, body.fixtures[k].shape.radius
    for o in test.gui_objects.values():  o['shape'] == 'circle', o['values'] = [centre, radius, colour]
    test.settings.drawShapes / drawAABBs

`export(env, e)` builds exactly those objects for ONE env of a batch from a ~1 KB device->host read; `build(...)`
does the same from numpy arrays (what the CPU tests drive).  Colours follow the reference: an agent listed in a
world contact is b2Color(1, 0.2, 0.2) (mvmnt.py:165-167), otherwise its base colour (mvmnt.py:21-22, or `colors[i]`,
mvmnt.py:68-69); TDM agents carry their team colour (combat.py:37-44) and dead ones are inactive bodies, which the
renderer dims by 3.  Targets are the white circles of radius `reward_radius` that mvmnt.py:54-57 puts into
`gui_objects`.  (In binary reward mode the reference never turns a collided agent back from red -- reset_color is
only called on the linear branch, mvmnt.py:172-175; this export always shows the current step's contacts.)

The same picture drawn on the device, for many envs at once: `BatchedFlock.render` / `BatchedTDM.render` (macm_render)
take the colours of `palette(env)` and the per-frame views of `fit_views`; `write_gif` turns frames into an animation.
"""
import numpy as np


class Color(object):
    """b2Color: r, g, b attributes, division by a scalar, iteration."""

    def __init__(self, r, g, b):
        self.r, self.g, self.b = float(r), float(g), float(b)

    def __truediv__(self, k):
        return Color(self.r / k, self.g / k, self.b / k)

    __div__ = __truediv__

    def __iter__(self):
        return iter((self.r, self.g, self.b))

    def __eq__(self, other):
        return tuple(self) == tuple(other)

    def __repr__(self):
        return "Color(%g, %g, %g)" % (self.r, self.g, self.b)


class Vec2(tuple):
    """b2Vec2 as the renderer uses it: indexable, .x / .y."""

    def __new__(cls, x, y):
        return tuple.__new__(cls, (float(x), float(y)))

    x = property(lambda self: self[0])
    y = property(lambda self: self[1])


class Transform(object):
    def __init__(self, position, angle):
        self.position, self.angle = position, float(angle)


class CircleShape(object):
    childCount = 1

    def __init__(self, radius):
        self.radius = float(radius)


class Fixture(object):
    def __init__(self, shape):
        self.shape = shape


class AgentData(object):
    """body.userData: the agent record (id, colour)."""

    def __init__(self, ID, color):
        self.id, self.color = ID, color


class Body(object):
    def __init__(self, transform, userData, radius, active=True, awake=True, velocity=(0.0, 0.0)):
        self.transform, self.userData = transform, userData
        self.position, self.angle = transform.position, transform.angle
        self.linearVelocity = Vec2(*velocity)
        self.active, self.awake = bool(active), bool(awake)
        self.fixtures = [Fixture(CircleShape(radius))]


class World(object):
    def __init__(self, bodies):
        self.bodies = bodies


class Frame(object):
    """What `PygletDraw(test)` reads from `test`: .world.bodies, .gui_objects, .settings."""

    def __init__(self, world, gui_objects, settings):
        self.world, self.gui_objects, self.settings = world, gui_objects, settings


FLOCK_BASE, COLLIDED, WHITE = (0.4, 0.4, 0.6), (1.0, 0.2, 0.2), (1.0, 1.0, 1.0)
TEAM_COLORS = ((0.2, 0.2, 1.0), (1.0, 0.2, 0.2), (0.2, 1.0, 0.2))   # combat.py:37-44


def build(posvel, angle, collided, settings, targets=None, colors=None, teams=None, alive=None, sleeping=None):
    """numpy state of ONE env -> Frame.  posvel [N,4], angle [N], collided [N]; Flock: targets [T,2];
    TDM: teams [N], alive [N]."""
    posvel = np.asarray(posvel, np.float64)
    N = posvel.shape[0]
    radius = settings.bodySettings["fixtures"].radius
    bodies = []
    for i in range(N):
        if teams is not None:
            t = int(teams[i])
            col = Color(*TEAM_COLORS[t]) if t < len(TEAM_COLORS) else None   # combat.py:37-44 has three teams
            ID = None
        else:
            base = colors[i] if colors else FLOCK_BASE
            col = Color(*COLLIDED) if collided[i] else Color(*base)
            ID = i
        act = True if alive is None else bool(alive[i])
        awake = True if sleeping is None else not bool(sleeping[i])
        bodies.append(Body(Transform(Vec2(posvel[i, 0], posvel[i, 1]), angle[i]), AgentData(i if ID is None else ID, col),
                           radius, active=act, awake=awake, velocity=(posvel[i, 2], posvel[i, 3])))
    gui = {}
    if targets is not None:
        for t, p in enumerate(np.asarray(targets, np.float64).reshape(-1, 2)):
            gui["target" + str(t)] = {"shape": "circle",
                                      "values": [Vec2(p[0], p[1]), settings.reward_radius, Color(*WHITE)]}
    return Frame(World(bodies), gui, settings)


def export(env, e=0):
    """One env of a BatchedFlock / BatchedTDM -> Frame (device->host read of that env's rows)."""
    t = env.engine.t
    posvel = t["posvel"][e].cpu().numpy()
    angle = t["angsleep"][e, :, 0].cpu().numpy()
    collided = t["collided"][e].cpu().numpy()
    if "tdm_state" in t:
        alive = (t["tdm_state"][e, :, 3].cpu().numpy().view(np.int32) & 1).astype(bool)
        return build(posvel, angle, collided, env.settings, teams=env.teams, alive=alive)
    return build(posvel, angle, collided, env.settings, targets=t["targets"][e].cpu().numpy(), colors=env.colors)


OTHER_TEAM = (0.5, 0.5, 0.5)   # teams beyond the three colours of combat.py:37-44


def _byte(c):
    return min(255, max(0, int(np.floor(255.0 * c + 0.5))))


def palette(env):
    """uint8 [N,2,3]: per agent the RGB bytes of its normal colour and of its alternate one, as `build` colours them --
    Flock: `colors[i]` or FLOCK_BASE, alternate (collided) COLLIDED; TDM: the team colour, alternate (dead) that colour
    / 3.  byte(c) = floor(255 c + 0.5), clamped to 0..255."""
    teams = getattr(env, "teams", None)
    N = len(teams) if teams is not None else sum(env.n_agents)
    pal = np.zeros((N, 2, 3), np.uint8)
    for i in range(N):
        if teams is not None:
            t = int(teams[i])
            col = Color(*(TEAM_COLORS[t] if t < len(TEAM_COLORS) else OTHER_TEAM))
            alt = col / 3
        else:
            col, alt = Color(*(env.colors[i] if env.colors else FLOCK_BASE)), Color(*COLLIDED)
        pal[i, 0] = [_byte(c) for c in col]
        pal[i, 1] = [_byte(c) for c in alt]
    return pal


def env_index(env, envs):
    """`envs` of a render call -> (int32 index tensor on the device, or None for every env; number of frames).
    A list, range or host array is checked on the host; a CUDA tensor costs one host synchronisation to check."""
    import torch
    E = env.engine.E
    if envs is None:
        return None, E
    if torch.is_tensor(envs):
        if envs.dtype.is_floating_point or envs.dtype == torch.bool or envs.dim() != 1:
            raise ValueError("envs must be a 1-D integer tensor")
        idx = envs
    else:
        a = np.asarray(list(envs) if isinstance(envs, range) else envs)
        if a.ndim != 1 or (a.size and a.dtype.kind not in "iu"):
            raise ValueError("envs must be a 1-D list of env indices")
        idx = torch.from_numpy(a.astype(np.int64))
    if idx.numel() == 0:
        raise ValueError("envs selects no env")
    if bool(((idx < 0) | (idx >= E)).any()):
        raise ValueError("envs holds an index outside 0..%d" % (E - 1))
    return idx.to(device=env.device, dtype=torch.int32).contiguous(), int(idx.numel())


def fit_views(env, envs, size):
    """float32 [B,3] views (centre x, centre y, half-width in metres), one per env of `envs` (None = every env), on the
    device of the env's state and without a host synchronisation: the smallest frame of aspect W / H = size[1] /
    size[0] that holds every agent's circle and, for Flock, every target circle, widened by 5 %."""
    import torch
    t = env.state
    H, W = int(size[0]), int(size[1])
    pos = t["posvel"][..., 0:2]
    if envs is not None:
        idx = envs if torch.is_tensor(envs) else torch.as_tensor(list(envs), dtype=torch.long)
        pos = pos.index_select(0, idx.to(device=pos.device, dtype=torch.long))
    r = float(env.settings.bodySettings["fixtures"].radius)
    lo, hi = (pos - r).amin(1), (pos + r).amax(1)
    if "targets" in t:
        tg = t["targets"]
        if envs is not None:
            tg = tg.index_select(0, idx.to(device=tg.device, dtype=torch.long))
        R = float(env.settings.reward_radius)
        lo, hi = torch.minimum(lo, (tg - R).amin(1)), torch.maximum(hi, (tg + R).amax(1))
    centre, half = (lo + hi) * 0.5, (hi - lo) * 0.5
    hw = torch.maximum(half[:, 0], half[:, 1] * (W / H)) * 1.05
    return torch.stack([centre[:, 0], centre[:, 1], hw], 1).to(torch.float32).contiguous()


def check_views(views, n_frames, device):
    """Caller-given views -> float32 [B,3] on the device.  A half-width that is not a finite value > 0 raises; checking
    a CUDA tensor costs one host synchronisation."""
    import torch
    v = torch.as_tensor(views, dtype=torch.float32)
    if tuple(v.shape) != (n_frames, 3):
        raise ValueError("views must be [%d, 3] (centre x, centre y, half-width), got %s" % (n_frames, tuple(v.shape)))
    hw = v[:, 2]
    if not bool((torch.isfinite(hw) & (hw > 0)).all()):
        raise ValueError("every view needs a finite half-width > 0")
    return v.to(device).contiguous()


def write_gif(frames, path, fps=30):
    """An animated GIF (looping) of uint8 frames [T,H,W,3] -- a numpy array or a tensor -- at `fps` frames per second.
    GIF stores at most 256 colours per frame: a frame with more (many agents with their own `colors` show up to four
    shades each) is quantised by PIL, and then reads back with slightly different colours."""
    try:
        from PIL import Image
    except ImportError as e:
        raise ImportError("write_gif needs PIL (the `pillow` package)") from e
    if hasattr(frames, "detach"):
        frames = frames.detach().cpu().numpy()
    a = np.asarray(frames)
    if a.ndim != 4 or a.shape[-1] != 3 or a.dtype != np.uint8 or a.shape[0] < 1:
        raise ValueError("frames must be uint8 [T,H,W,3], got %s %s" % (a.dtype, a.shape))
    imgs = [Image.fromarray(f, "RGB") for f in a]
    imgs[0].save(path, save_all=True, append_images=imgs[1:], duration=max(1, int(round(1000.0 / fps))), loop=0)
