"""The drawing rules of macm_render (include/macm.h), restated in float64 numpy from the objects the reference's renderer
reads (a gym_macm.render Frame, walked in the order of `_manual_draw` in test_render_cpu.py), with known answers; the
colours, views and GIF writer of gym_macm.render.  No GPU: tests/test_gpu_render.py holds the kernel to `rasterize`."""
import os
import re
import types

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EPS_D2 = 1e-3     # px^2: a disc or ring pixel this close to its threshold may go either way in the kernel
EPS_AXIS = 1e-3   # px: the same for the distance to the heading axis


def _byte(c):
    return min(255, max(0, int(np.floor(255.0 * c + 0.5))))


def rasterize(frame, view, size):
    """float64 frame of a render.build Frame: (uint8 [H,W,3], bool [H,W] ambiguous pixels).  `view` is (cx, cy, hw)
    as the float32 values the kernel reads; size = (H, W)."""
    H, W = int(size[0]), int(size[1])
    img = np.zeros((H, W, 3), np.uint8)
    amb = np.zeros((H, W), bool)
    cx, cy, hw = (float(np.float32(x)) for x in view)
    if not (np.isfinite(hw) and hw > 0):
        return img, amb
    s = W / (2.0 * hw)
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

    for body in frame.world.bodies:
        col = body.userData.color
        col = tuple(col) if col is not None else (0.5, 0.5, 0.5)   # teams beyond combat.py's three
        if not body.active:
            col = tuple(c / 3 for c in col)
        rgb = np.array([_byte(c) for c in col], np.uint8)
        x, y = body.transform.position
        u, v = (x - cx) * s + W / 2, (cy - y) * s + H / 2
        rho = body.fixtures[0].shape.radius * s
        r = region(u, v, rho + 1.0)
        if r is None:
            continue
        sl, dx, dy = r
        d2 = dx * dx + dy * dy
        img[sl][d2 <= rho * rho] = rgb >> 1                            # the disc at half the colour
        outline, near = ring(d2, rho)
        img[sl][outline] = rgb
        ux, uy = np.cos(body.transform.angle), -np.sin(body.transform.angle)
        t = np.clip(dx * ux + dy * uy, 0.0, rho)
        ex, ey = dx - t * ux, dy - t * uy
        dist2 = ex * ex + ey * ey
        img[sl][dist2 <= 0.25] = rgb                                   # the heading axis
        amb[sl] |= near | (np.abs(np.sqrt(dist2) - 0.5) < EPS_AXIS)
    for obj in frame.gui_objects.values():
        if obj["shape"] != "circle":
            continue
        c, rad, col = obj["values"]
        u, v = (c[0] - cx) * s + W / 2, (cy - c[1]) * s + H / 2
        rho = rad * s
        r = region(u, v, rho + 1.0)
        if r is None:
            continue
        sl, dx, dy = r
        d2 = dx * dx + dy * dy
        hit, near = ring(d2, rho)
        img[sl][hit] = np.array([_byte(k) for k in col], np.uint8)
        amb[sl] |= near
    return img, amb


# ---- known answers ---------------------------------------------------------------------------------------------
def _flock_frame(pos, angle, collided=None, targets=None, colors=None, **kw):
    from gym_macm import render
    from gym_macm.settings import flockSettings
    pos = np.asarray(pos, np.float32).reshape(-1, 2)
    n = len(pos)
    posvel = np.zeros((n, 4), np.float32)
    posvel[:, 0:2] = pos
    coll = np.zeros(n, np.uint8) if collided is None else np.asarray(collided, np.uint8)
    return render.build(posvel, np.asarray(angle, np.float32), coll, flockSettings(**kw), targets=targets, colors=colors)


BASE, RED = np.array([102, 102, 153]), np.array([255, 51, 51])    # FLOCK_BASE, COLLIDED in bytes
# 12 x 12 pixels at 6 px per metre (exact in float32): an agent of radius 0.5 m at the origin has rho = 3 px and its
# centre on the centre of pixel (4, 4)
S6, SIZE = (0.25, -0.25, 1.0), (12, 12)


def _classes(img, rgb):
    col = (img == rgb).all(-1)
    fill = (img == rgb >> 1).all(-1)
    return col, fill, (img == 0).all(-1)


def test_disc_at_a_pixel_centre():
    img, amb = rasterize(_flock_frame([[0, 0]], [0.0]), S6, SIZE)
    col, fill, bg = _classes(img, BASE)
    # 29 pixel centres within 3 px; outline 4 < d^2 <= 9: 16 of them; the axis adds (4,4) (4,5) (4,6)
    assert (col.sum(), fill.sum(), bg.sum()) == (19, 10, 144 - 29)
    assert col[4, 4:8].all() and not col[4, 8] and fill[3, 4] and fill[4, 3]
    # centres exactly on the outer (d^2 = 9: 4 pixels) or inner (d^2 = 4: 4 pixels) threshold are the ambiguous ones
    assert amb.sum() == 8 and amb[4, 7] and amb[2, 4] and amb[4, 1]


@pytest.mark.parametrize("theta,pixels", [(0.0, [(4, 4), (4, 5), (4, 6), (4, 7)]),
                                          (np.pi / 2, [(4, 4), (3, 4), (2, 4), (1, 4)]),
                                          (-np.pi / 2, [(4, 4), (5, 4), (6, 4), (7, 4)])])
def test_axis_direction(theta, pixels):
    img, _ = rasterize(_flock_frame([[0, 0]], [theta]), S6, SIZE)
    col, fill, _ = _classes(img, BASE)
    axis = {(i, j) for i, j in zip(*np.nonzero(col)) if (i - 4) ** 2 + (j - 4) ** 2 <= 4}   # inside the outline
    assert axis == set(pixels[:3])
    assert col[pixels[3]]   # the tip lies on the outline
    # +y is up: angle pi/2 points at row 0
    opposite = (8 - pixels[2][0], 8 - pixels[2][1])
    assert fill[opposite]


def test_higher_index_paints_over_lower():
    # agent 0 at column 4, agent 1 (collided) at column 7, both facing -x: their discs overlap
    img, _ = rasterize(_flock_frame([[0, 0], [0.5, 0]], [np.pi, np.pi], collided=[0, 1]), S6, SIZE)
    assert (img[3, 6] == RED >> 1).all()      # agent 1's fill over agent 0's outline
    assert (img[4, 4] == RED).all()           # agent 1's axis tip over agent 0's axis
    assert (img[4, 1] == BASE).all() and (img[3, 3] == BASE >> 1).all()
    img, _ = rasterize(_flock_frame([[0.5, 0], [0, 0]], [np.pi, np.pi], collided=[1, 0]), S6, SIZE)
    assert (img[3, 6] == BASE).all()          # swapped: the base agent's outline now on top
    assert (img[4, 4] == BASE).all()


def test_target_ring_over_agents():
    # a ring of the agent's own radius around it
    fr = _flock_frame([[0, 0]], [0.0], targets=np.array([[0.0, 0.0]], np.float32), _reward_radius=0.5)
    img, _ = rasterize(fr, S6, SIZE)
    white, _, _ = _classes(img, np.array([255, 255, 255]))
    col, fill, _ = _classes(img, BASE)
    assert white.sum() == 16 and col.sum() == 3 and fill.sum() == 10   # the ring replaces the outline, not the fill


def test_off_frame_agent_draws_nothing():
    img, amb = rasterize(_flock_frame([[10, 0], [0, -2.2]], [0.0, 1.0]), S6, SIZE)
    assert not img.any() and not amb.any()


def test_agent_larger_than_the_frame_fills_it():
    img, _ = rasterize(_flock_frame([[0, 0]], [0.0]), (0.0075, -0.0075, 0.03), SIZE)   # rho = 100 px, centre (4, 4)
    col, fill, bg = _classes(img, BASE)
    assert not bg.any() and col.sum() == 8 and col[4, 4:].all() and fill.sum() == 144 - 8


def test_bad_view_is_background():
    fr = _flock_frame([[0, 0]], [0.0])
    for v in ((0, 0, 0.0), (0, 0, -1.0), (0, 0, np.inf), (0, 0, np.nan)):
        img, _ = rasterize(fr, v, (11, 11))
        assert not img.any()


# ---- colours, views, GIFs --------------------------------------------------------------------------------------
def test_flock_palette():
    from gym_macm import render
    env = types.SimpleNamespace(n_agents=[2, 1], colors=None)
    p = render.palette(env)
    assert p.dtype == np.uint8 and p.shape == (3, 2, 3)
    assert (p[:, 0] == BASE).all() and (p[:, 1] == RED).all()
    env = types.SimpleNamespace(n_agents=[2], colors=[(0, 1, 0), (0.5, 0.25, 1.2)])
    p = render.palette(env)
    assert p[0, 0].tolist() == [0, 255, 0] and p[1, 0].tolist() == [128, 64, 255] and (p[:, 1] == RED).all()


def test_tdm_palette():
    from gym_macm import render
    env = types.SimpleNamespace(teams=[0, 0, 1, 2, 3])
    p = render.palette(env)
    assert p[:, 0].tolist() == [[51, 51, 255], [51, 51, 255], [255, 51, 51], [51, 255, 51], [128, 128, 128]]
    assert p[:, 1].tolist() == [[17, 17, 85], [17, 17, 85], [85, 17, 17], [17, 85, 17], [43, 43, 43]]


def test_palette_is_the_colour_the_restatement_draws():
    """Frame colours (render.build, dimmed by the renderer for dead agents) == palette bytes (normal / alternate)."""
    from gym_macm import render
    from gym_macm.settings import combatSettings
    teams, alive = [0, 1, 2, 3], [1, 0, 1, 0]
    fr = render.build(np.zeros((4, 4), np.float32), np.zeros(4), np.zeros(4, np.uint8), combatSettings(), teams=teams,
                      alive=alive)
    p = render.palette(types.SimpleNamespace(teams=teams))
    for i, b in enumerate(fr.world.bodies):
        c = tuple(b.userData.color) if b.userData.color is not None else (0.5, 0.5, 0.5)
        c = c if b.active else tuple(x / 3 for x in c)
        assert [_byte(x) for x in c] == p[i, 0 if alive[i] else 1].tolist()


@pytest.mark.parametrize("size", [(84, 84), (480, 640), (64, 32)])
def test_fit_views(size):
    import torch
    from gym_macm import render
    from gym_macm.settings import flockSettings
    H, W = size
    posvel = torch.zeros((3, 2, 4))
    posvel[0, :, 0:2] = torch.tensor([[0.0, 0.0], [10.0, 2.0]])
    posvel[1, :, 0:2] = torch.tensor([[-1.0, 5.0], [-1.0, -5.0]])
    posvel[2, :, 0:2] = torch.tensor([[3.0, 3.0], [3.0, 3.0]])
    targets = torch.tensor([[[0.0, 0.0]], [[0.0, 0.0]], [[40.0, 3.0]]])
    env = types.SimpleNamespace(state={"posvel": posvel, "targets": targets}, settings=flockSettings(reward_radius=7.0))
    v = render.fit_views(env, None, size)
    assert v.dtype == torch.float32 and tuple(v.shape) == (3, 3)
    # env 0: x in [-7, 10.5], y in [-7, 7]; env 1: x in [-7, 7], y in [-7, 7]; env 2: x in [2.5, 47], y in [-4, 10]
    boxes = [(-7.0, 10.5, -7.0, 7.0), (-7.0, 7.0, -7.0, 7.0), (2.5, 47.0, -4.0, 10.0)]
    for k, (x0, x1, y0, y1) in enumerate(boxes):
        hw = max((x1 - x0) / 2, (y1 - y0) / 2 * W / H) * 1.05
        assert np.allclose(v[k].numpy(), [(x0 + x1) / 2, (y0 + y1) / 2, hw], rtol=1e-6)
    # the frame holds the box: half-height hw * H / W covers the y extent
    assert (v[:, 2] * H / W >= torch.tensor([b[3] - b[2] for b in boxes]) / 2).all()
    sub = render.fit_views(env, [2, 0, 2], size)
    assert torch.equal(sub, v[[2, 0, 2]])
    # TDM: no targets
    env = types.SimpleNamespace(state={"posvel": posvel}, settings=flockSettings())
    v = render.fit_views(env, None, size)
    assert np.allclose(v[1].numpy(), [-1.0, 0.0, max(0.5, 5.5 * W / H) * 1.05], rtol=1e-6)


def test_write_gif_round_trip(tmp_path):
    from PIL import Image
    from gym_macm import render
    rng = np.random.default_rng(0)
    colours = np.array([[0, 0, 0], [102, 102, 153], [51, 51, 76], [255, 51, 51], [255, 255, 255]], np.uint8)
    frames = colours[rng.integers(0, len(colours), (3, 24, 40))]
    path = str(tmp_path / "flock.gif")
    render.write_gif(frames, path, fps=20)
    im = Image.open(path)
    assert im.n_frames == 3
    for k in range(3):
        im.seek(k)
        assert np.array_equal(np.asarray(im.convert("RGB")), frames[k])
    with pytest.raises(ValueError):
        render.write_gif(frames[..., 0], path)


def test_render_args_layout_matches_header():
    from gym_macm import _lib
    hdr = open(os.path.join(ROOT, "include", "macm.h")).read()
    body = hdr[hdr.index("typedef struct macm_render_args {"):hdr.index("} macm_render_args;")]
    names = []
    for line in body.splitlines()[1:]:
        m = re.match(r"\s*(?:const\s+)?(?:int32_t|float|uint8_t)\*?\s+([^;]+);", line.split("/*")[0])
        if m:
            names += [n.strip().lstrip("*") for n in m.group(1).split(",")]
    assert names == [f[0] for f in _lib.MacmRenderArgs._fields_]
