"""The drawing rules of macm_render_agents (include/macm.h), restated in float64 numpy from the objects the reference's
renderer reads (a gym_macm.render Frame), with known answers: every agent's own frame, centred on it with its heading
up.  The ambiguity bands are those of test_raster_cpu.  No GPU: tests/test_gpu_agent_frames.py holds the kernel to
`rasterize_agent`."""
import math
import os
import re
import types

import numpy as np
import pytest

from test_raster_cpu import BASE, EPS_AXIS, EPS_D2, RED, _byte, _flock_frame

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def project(frame, i, half_width, size):
    """Pixel centres (u, v) of every agent then every target in the frame of agent i, and the scale s in px / m."""
    H, W = int(size[0]), int(size[1])
    s = W / (2.0 * half_width)
    obs = frame.world.bodies[i]
    cx, cy = obs.transform.position
    ci, si = np.cos(obs.transform.angle), np.sin(obs.transform.angle)
    pts = [b.transform.position for b in frame.world.bodies]
    pts += [o["values"][0] for o in frame.gui_objects.values() if o["shape"] == "circle"]
    uv = []
    for x, y in pts:
        dx, dy = x - cx, y - cy
        uv.append((W / 2 + s * (dx * si - dy * ci), H / 2 - s * (dx * ci + dy * si)))
    return np.array(uv, np.float64).reshape(-1, 2), s


def rasterize_agent(frame, i, half_width, size):
    """float64 frame of agent i of a render.build Frame: (uint8 [H,W,3], bool [H,W] ambiguous pixels)."""
    H, W = int(size[0]), int(size[1])
    img = np.zeros((H, W, 3), np.uint8)
    amb = np.zeros((H, W), bool)
    uv, s = project(frame, i, half_width, size)
    a = frame.world.bodies[i].transform.angle
    ci, si = np.cos(a), np.sin(a)
    pxs, pys = np.arange(W) + 0.5, np.arange(H) + 0.5

    def region(u, v, reach):
        # the pixels a primitive of centre (u, v) can cover; everything else keeps what it has
        if not (np.isfinite(u) and np.isfinite(v)):
            return None
        j0, j1 = max(0, int(np.floor(u - reach)) - 1), min(W, int(np.ceil(u + reach)) + 1)
        i0, i1 = max(0, int(np.floor(v - reach)) - 1), min(H, int(np.ceil(v + reach)) + 1)
        if j0 >= j1 or i0 >= i1:
            return None
        sl = (slice(i0, i1), slice(j0, j1))
        return sl, pxs[sl[1]][None, :] - u, pys[sl[0]][:, None] - v

    def ring(d2, rho):
        r2, in2 = rho * rho, (rho - 1.0) * (rho - 1.0)
        near = np.abs(d2 - r2) < EPS_D2
        if rho >= 1.0:
            near |= np.abs(d2 - in2) < EPS_D2
        return (d2 <= r2) & ((rho < 1.0) | (d2 > in2)), near

    bodies = frame.world.bodies
    for k, body in enumerate(bodies):
        col = body.userData.color
        col = tuple(col) if col is not None else (0.5, 0.5, 0.5)   # teams beyond combat.py's three
        if not body.active:
            col = tuple(c / 3 for c in col)
        rgb = np.array([_byte(c) for c in col], np.uint8)
        rho = body.fixtures[0].shape.radius * s
        r = region(uv[k, 0], uv[k, 1], rho + 1.0)
        if r is None:
            continue
        sl, dx, dy = r
        d2 = dx * dx + dy * dy
        img[sl][d2 <= rho * rho] = rgb >> 1                            # the disc at half the colour
        outline, near = ring(d2, rho)
        img[sl][outline] = rgb
        ck, sk = np.cos(body.transform.angle), np.sin(body.transform.angle)
        ux, uy = ck * si - sk * ci, -(ck * ci + sk * si)
        t = np.clip(dx * ux + dy * uy, 0.0, rho)
        ex, ey = dx - t * ux, dy - t * uy
        dist2 = ex * ex + ey * ey
        img[sl][dist2 <= 0.25] = rgb                                   # the heading axis
        amb[sl] |= near | (np.abs(np.sqrt(dist2) - 0.5) < EPS_AXIS)
    k = len(bodies)
    for obj in frame.gui_objects.values():
        if obj["shape"] != "circle":
            continue
        _, rad, col = obj["values"]
        rho = rad * s
        r = region(uv[k, 0], uv[k, 1], rho + 1.0)
        k += 1
        if r is None:
            continue
        sl, dx, dy = r
        d2 = dx * dx + dy * dy
        hit, near = ring(d2, rho)
        img[sl][hit] = np.array([_byte(c) for c in col], np.uint8)
        amb[sl] |= near
    return img, amb


def agent_frames(frames, envs, half_width, size):
    """Frames [B,N,H,W,3] and ambiguity [B,N,H,W] of the envs `frames` (a Frame per env) at rows `envs`; an index
    outside [0, len(frames)) gives N black frames."""
    N = len(frames[0].world.bodies)
    H, W = int(size[0]), int(size[1])
    img = np.zeros((len(envs), N, H, W, 3), np.uint8)
    amb = np.zeros((len(envs), N, H, W), bool)
    for b, e in enumerate(envs):
        if 0 <= e < len(frames):
            for i in range(N):
                img[b, i], amb[b, i] = rasterize_agent(frames[e], i, half_width, size)
    return img, amb


# ---- known answers ---------------------------------------------------------------------------------------------
# an odd frame puts the observer's centre on the centre of pixel (6, 6); 6 px per metre gives a 0.5 m agent rho = 3 px
SIZE13, HW13 = (13, 13), 13 / 12.0
ANGLES = [0.0, np.pi, -np.pi, np.pi / 2, -np.pi / 2, 1.0, 2.5, -3.0]


def _classes(img, rgb):
    return (img == rgb).all(-1), (img == rgb >> 1).all(-1), (img == 0).all(-1)


@pytest.mark.parametrize("theta", ANGLES)
def test_observer_centred_heading_up(theta):
    fr = _flock_frame([[1.25, -0.5]], [theta])
    uv, s = project(fr, 0, HW13, SIZE13)
    assert s == 6.0 and tuple(uv[0]) == (6.5, 6.5)
    img, amb = rasterize_agent(fr, 0, HW13, SIZE13)
    col, fill, bg = _classes(img, BASE)
    # what the top-down frame of an agent at angle pi/2 shows (test_raster_cpu.test_disc_at_a_pixel_centre, turned)
    assert (col.sum(), fill.sum(), bg.sum()) == (19, 10, 169 - 29)
    axis = {(r, c) for r, c in zip(*np.nonzero(col)) if (r - 6) ** 2 + (c - 6) ** 2 <= 4}   # inside the outline
    assert axis == {(6, 6), (5, 6), (4, 6)} and col[3, 6] and fill[8, 6]
    # the frame is mirror-symmetric about the heading axis
    ok = ~(amb | amb[:, ::-1])
    assert (img[ok] == img[:, ::-1][ok]).all()


@pytest.mark.parametrize("theta", ANGLES)
def test_neighbours_ahead_and_to_the_right(theta):
    c, a = np.array([0.75, -1.5]), np.float32(theta)
    h = np.array([np.cos(float(a)), np.sin(float(a))])
    right = np.array([h[1], -h[0]])
    pos = [c, c + 2 * h, c + 2 * right]
    colors = [(1, 1, 1), (0, 1, 0), (0, 0, 1)]
    fr = _flock_frame(pos, [theta, 0.3, -2.0], colors=colors)
    size, hw = (41, 41), 41 / 12.0
    uv, s = project(fr, 0, hw, size)
    assert s == 6.0
    # float32 positions: within 1e-5 px of the exact answer
    assert np.abs(uv - [[20.5, 20.5], [20.5, 20.5 - 2 * s], [20.5 + 2 * s, 20.5]]).max() < 1e-5
    img, _ = rasterize_agent(fr, 0, hw, size)
    assert img[8, 20].tolist() == [0, 255, 0]     # the centre of the neighbour ahead: its heading axis
    assert img[20, 32].tolist() == [0, 0, 255]    # the one to the right


@pytest.mark.parametrize("phi", [0.7, -2.0, np.pi])
@pytest.mark.parametrize("i", [0, 3])
def test_rotating_the_world_about_the_observer_keeps_its_frame(phi, i):
    rng = np.random.default_rng(7)
    pos = rng.uniform(-3, 3, (8, 2)).astype(np.float32)
    ang = rng.uniform(-np.pi, np.pi, 8).astype(np.float32)
    coll = rng.integers(0, 2, 8)
    tg = rng.uniform(-3, 3, (2, 2)).astype(np.float32)
    size, hw = (48, 40), 4.0

    def turned(p):
        d = p.astype(np.float64) - pos[i]
        cp, sp = np.cos(phi), np.sin(phi)
        return (pos[i] + np.stack([cp * d[:, 0] - sp * d[:, 1], sp * d[:, 0] + cp * d[:, 1]], 1)).astype(np.float32)

    kw = dict(collided=coll, _reward_radius=1.5)
    a, amb_a = rasterize_agent(_flock_frame(pos, ang, targets=tg, **kw), i, hw, size)
    b, amb_b = rasterize_agent(_flock_frame(turned(pos), (ang + phi).astype(np.float32), targets=turned(tg), **kw),
                               i, hw, size)
    assert len(np.unique(a.reshape(-1, 3), axis=0)) >= 4, "the frame should show other agents or targets"
    ok = ~(amb_a | amb_b)
    assert (a[ok] == b[ok]).all()
    assert amb_a.mean() < 0.02


def test_target_rings():
    # a ring of the agent's own radius around the observer replaces its outline, not its fill
    fr = _flock_frame([[0, 0]], [0.4], targets=np.array([[0.0, 0.0]], np.float32), _reward_radius=0.5)
    img, _ = rasterize_agent(fr, 0, HW13, SIZE13)
    white, _, _ = _classes(img, np.array([255, 255, 255]))
    col, fill, _ = _classes(img, BASE)
    assert white.sum() == 16 and col.sum() == 3 and fill.sum() == 10
    # a target 1.5 m behind the observer (facing -y): a ring of radius 6 px centred 9 px below the frame's centre
    fr = _flock_frame([[0, 0]], [-np.pi / 2], targets=np.array([[0.0, 1.5]], np.float32), _reward_radius=1.0)
    size = (41, 41)
    img, amb = rasterize_agent(fr, 0, 41 / 12.0, size)
    white, _, _ = _classes(img, np.array([255, 255, 255]))
    r, c = np.nonzero(white & ~amb)
    d2 = (r + 0.5 - 29.5) ** 2 + (c + 0.5 - 20.5) ** 2
    assert len(r) > 20 and (d2 <= 36).all() and (d2 > 25).all()


def test_higher_index_paints_over_lower():
    # observer 0 facing world +y: its frame is the world's axes.  Agent 1 (collided) 0.5 m to its right, both
    # facing -x: their discs overlap
    img, _ = rasterize_agent(_flock_frame([[0, 0], [0.5, 0]], [np.pi / 2, np.pi], collided=[0, 1]), 0, HW13, SIZE13)
    assert (img[5, 8] == RED >> 1).all()      # agent 1's fill over agent 0's outline
    assert (img[6, 6] == RED).all()           # agent 1's axis tip over agent 0's axis
    assert (img[6, 3] == BASE).all() and (img[5, 5] == BASE >> 1).all()
    img, _ = rasterize_agent(_flock_frame([[0.5, 0], [0, 0]], [np.pi, np.pi / 2], collided=[1, 0]), 1, HW13, SIZE13)
    assert (img[5, 8] == BASE).all()          # swapped: the base agent's outline now on top
    assert (img[6, 6] == BASE).all()


def test_dead_agent_keeps_its_frame():
    from gym_macm import render
    from gym_macm.settings import combatSettings
    posvel = np.zeros((2, 4), np.float32)
    posvel[1, 0] = 1.0
    fr = render.build(posvel, np.float32([0.0, 2.0]), np.zeros(2, np.uint8), combatSettings(), teams=[0, 1],
                      alive=[0, 1])
    img, _ = rasterize_agent(fr, 0, HW13, SIZE13)
    assert img[6, 6].tolist() == [17, 17, 85]     # the dead observer, in a third of its team colour
    assert img[0, 6].tolist() == [255, 51, 51]    # the live agent 1 m ahead of it


def test_bad_env_rows_are_black():
    rng = np.random.default_rng(3)
    frames = [_flock_frame(rng.uniform(-2, 2, (4, 2)), rng.uniform(-3, 3, 4)) for _ in range(2)]
    img, amb = agent_frames(frames, [1, -1, 2, 0, 1], 3.0, (16, 16))
    assert img.shape == (5, 4, 16, 16, 3)
    assert not img[1].any() and not img[2].any() and not amb[1].any() and not amb[2].any()
    assert img[0].any() and img[3].any() and np.array_equal(img[0], img[4])


def test_python_rejects_bad_arguments_before_the_call():
    from gym_macm import batched
    fake = types.SimpleNamespace()   # fails on any use: the checks come first
    for size, hw in (((0, 16), 1.0), ((16, 1025), 1.0), ((1025, 16), 1.0), ((16, 16), 0.0), ((16, 16), -2.0),
                     ((16, 16), math.inf), ((16, 16), math.nan)):
        with pytest.raises(ValueError):
            batched._BatchedCommon.render_agents(fake, size, hw)


def test_agent_frames_args_layout_matches_header():
    from gym_macm import _lib
    hdr = open(os.path.join(ROOT, "include", "macm.h")).read()
    body = hdr[hdr.index("typedef struct macm_agent_frames_args {"):hdr.index("} macm_agent_frames_args;")]
    fields = []
    for line in body.splitlines()[1:]:
        m = re.match(r"\s*(?:const\s+)?(int32_t|double|uint8_t)(\*?)\s+([^;]+);", line.split("/*")[0])
        if m:
            kind = "ptr" if m.group(2) else m.group(1)
            fields += [(n.strip().lstrip("*"), kind) for n in m.group(3).split(",")]
    ctypes_kind = {_lib.i32: "int32_t", _lib.f64: "double"}
    assert fields == [(n, ctypes_kind.get(t, "ptr")) for n, t in _lib.MacmAgentFramesArgs._fields_]
    assert _lib.ABI_VERSION == int(re.search(r"#define MACM_ABI_VERSION (\d+)", hdr).group(1)) == 8
