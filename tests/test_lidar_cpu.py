"""Lidar scans (macm_lidar, include/macm.h) on the CPU.  The oracle's scan is its closest-hit ray cast
(`oracle_world_raycast`: ow_raycast_closest, the TDM attack's query) once per ray, from ray ends built by the rule
(float64 directions through libm, fp32 ends); it is held bit for bit to a vectorised numpy restatement of the whole
rule, with known answers.  Also the ctypes layout of macm_lidar_args and the Python argument checks.  No GPU:
tests/test_gpu_lidar.py holds the kernel to the oracle's scan."""
import math
import os
import re
import types

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
f32 = np.float32
EPS = f32(1.1920929e-07)   # b2_epsilon
_cos, _sin = np.frompyfunc(math.cos, 1, 1), np.frompyfunc(math.sin, 1, 1)   # libm, as the oracle


def ray_ends(pos, ang, n_rays, fov, max_range):
    """fp32 ray ends p2 [N,R,2] of every agent: th = a + fov (2r + 1 - R) / (2R) in float64, (float)(L cos th) added
    to the fp32 centre in fp32."""
    r = np.arange(n_rays)
    o = fov * ((2 * r + 1 - n_rays).astype(np.float64) / float(2 * n_rays))
    th = np.asarray(ang, f32).astype(np.float64)[:, None] + o[None, :]
    dx = (max_range * _cos(th).astype(np.float64)).astype(f32)
    dy = (max_range * _sin(th).astype(np.float64)).astype(f32)
    p = np.asarray(pos, f32)
    return np.stack([p[:, None, 0] + dx, p[:, None, 1] + dy], -1)


def scan(pos, ang, n_rays, fov, max_range, proxy=None, radius=0.5):
    """One env's scan: (fraction float32 [N,R], hit int32 [N,R]).  b2CircleShape::RayCast of every ray against every
    body with a proxy, in fp32 and Box2D's operation order; the smallest fraction, lowest index among equal ones."""
    p = np.asarray(pos, f32)
    N = len(p)
    proxy = np.ones(N, bool) if proxy is None else np.asarray(proxy, bool)
    rad = f32(radius)
    p2 = ray_ends(p, ang, n_rays, fov, max_range)
    p1 = p[:, None, None, :]                                  # [N,1,1,2]
    sx, sy = p1[..., 0] - p[None, None, :, 0], p1[..., 1] - p[None, None, :, 1]   # [N,1,M]
    bb = (sx * sx + sy * sy) - rad * rad
    rx, ry = (p2[..., 0] - p[:, None, 0])[..., None], (p2[..., 1] - p[:, None, 1])[..., None]   # [N,R,1]
    cq = sx * rx + sy * ry
    rr = rx * rx + ry * ry
    sigma = cq * cq - rr * bb
    ok = (sigma >= 0) & (rr >= EPS) & proxy[None, None, :]
    with np.errstate(invalid="ignore", divide="ignore"):
        a = -(cq + np.sqrt(np.where(ok, sigma, f32(0))))
        ok &= (f32(0) <= a) & (a <= rr)
        frac = np.where(ok, a / rr, f32(np.inf))
    k = np.argmin(frac, -1)                                   # the first of equal minima: the lowest index
    best = np.take_along_axis(frac, k[..., None], -1)[..., 0]
    hit = np.where(ok.any(-1), k, -1).astype(np.int32)
    return np.where(hit >= 0, best, f32(1)).astype(f32), hit


def world_scan(world, n_rays, fov, max_range):
    """The oracle's scan of one world (an OracleWorld): for every body and ray, the ray end of `ray_ends` and the
    oracle's closest-hit cast (`oracle_world_raycast`, ow_raycast_closest).  (fraction float32 [N,R], hit int32 [N,R])"""
    b = world.bodies()
    p2 = ray_ends(b[:, 0:2], b[:, 4], n_rays, fov, max_range)
    shape = (world.n, int(n_rays))
    fr, hit = np.ones(shape, f32), np.full(shape, -1, np.int32)
    for i in range(world.n):
        p1 = (float(b[i, 0]), float(b[i, 1]))
        for r in range(int(n_rays)):
            hit[i, r], fr[i, r] = world.raycast(p1, (float(p2[i, r, 0]), float(p2[i, r, 1])))
    return fr, hit


def make_world(pos, ang, dead=(), radius=0.5):
    from oracle import oracle
    w = oracle.OracleWorld(radius=radius)
    for (x, y), a in zip(pos, ang):
        w.add_body(x, y, a)
    for i in dead:
        w.set_active(i, 0)
    return w


def oracle_scan(pos, ang, n_rays, fov, max_range, proxy=None, radius=0.5):
    """The oracle's scan of one env given as fp32 positions [N,2], angles [N] and proxy bits [N] (None: all)."""
    dead = () if proxy is None else np.flatnonzero(~np.asarray(proxy, bool))
    return world_scan(make_world(np.asarray(pos, np.float64), np.asarray(ang, np.float64), dead, radius),
                      n_rays, fov, max_range)


def same_bits(a, b):
    return np.array_equal(np.asarray(a, f32).view(np.int32), np.asarray(b, f32).view(np.int32))


@pytest.mark.parametrize("N,R,fov,L,spread", [(6, 32, 2 * np.pi, 10.0, 8.0), (17, 33, np.pi, 4.0, 5.0),
                                              (40, 1, 0.3, 1e4, 20.0), (33, 7, 2 * np.pi, 0.01, 1.5),
                                              (64, 128, 1.0, 1.0, 6.0)])
def test_oracle_equals_numpy_restatement(N, R, fov, L, spread):
    rng = np.random.default_rng(N * 1000 + R)
    hits = 0
    for e in range(3):
        pos = (spread * (rng.random((N, 2)) - 0.5)).astype(f32)
        ang = rng.uniform(-8, 8, N).astype(f32)
        fr, hit = oracle_scan(pos, ang, R, fov, L)
        f2, h2 = scan(pos, ang, R, fov, L)
        assert same_bits(fr, f2) and np.array_equal(hit, h2)
        hits += int((h2 >= 0).sum())
    assert hits > 0


def test_oracle_equals_restatement_with_dead_agents():
    rng = np.random.default_rng(7)
    pos, ang = rng.uniform(-3, 3, (30, 2)), rng.uniform(-4, 4, 30)
    dead = [0, 3, 4, 11, 29]
    w = make_world(pos, ang, dead)
    fr, hit = world_scan(w, 64, 2 * np.pi, 8.0)
    b = w.bodies()
    proxy = np.ones(30, bool)
    proxy[dead] = False
    f2, h2 = scan(b[:, 0:2], b[:, 4], 64, 2 * np.pi, 8.0, proxy)
    assert same_bits(fr, f2) and np.array_equal(hit, h2)
    assert not np.isin(hit, dead).any() and (hit >= 0).sum() > 100
    assert (h2[dead] >= 0).any()   # dead agents still scan


def test_body_straight_ahead():
    # (3 - 0.5) / 10: s = (-3, 0), bb = 8.75, c = -30, rr = 100, sigma = 25, a = 25
    fr, hit = world_scan(make_world([(0, 0), (3, 0)], [0, 0]), 1, 2 * np.pi, 10.0)
    assert fr[0, 0] == f32(0.25) and hit[0, 0] == 1
    # and from a heading of pi / 2
    fr, hit = world_scan(make_world([(0, 0), (0, 3)], [np.pi / 2, 0]), 1, 1.0, 10.0)
    assert hit[0, 0] == 1 and abs(fr[0, 0] - 0.25) < 1e-6


def test_behind_and_beyond_reach_are_misses():
    fr, hit = world_scan(make_world([(0, 0), (-3, 0)], [0, 0]), 1, 0.5, 10.0)
    assert hit[0, 0] == -1 and fr[0, 0] == 1
    fr, hit = world_scan(make_world([(0, 0), (10.5 + 1e-3, 0)], [0, 0]), 1, 0.5, 10.0)
    assert hit[0, 0] == -1 and fr[0, 0] == 1
    fr, hit = world_scan(make_world([(0, 0), (10.4, 0)], [0, 0]), 1, 0.5, 10.0)
    assert hit[0, 0] == 1 and abs(fr[0, 0] - 0.99) < 2e-6


def test_tangent_ray():
    # the ray y = 0 touches the disc of radius 0.5 centred at (3, 0.5): sigma = 900 - 900 = 0, a = 30
    fr, hit = world_scan(make_world([(0, 0), (3, 0.5)], [0, 0]), 1, 0.5, 10.0)
    assert hit[0, 0] == 1 and fr[0, 0] == f32(0.3)
    fr, hit = world_scan(make_world([(0, 0), (3, 0.5001)], [0, 0]), 1, 0.5, 10.0)
    assert hit[0, 0] == -1 and fr[0, 0] == 1


def test_origin_inside_a_neighbour():
    # agent 0 sits inside agent 1's disc: no ray reports 1 (or 0 itself), and the ray ahead still reaches agent 2
    w = make_world([(0, 0), (0.2, 0.1), (3, 0)], [0, 0, 0])
    fr, hit = world_scan(w, 16, 2 * np.pi, 10.0)
    assert not (hit[0] == 1).any() and not (hit[0] == 0).any()
    fr, hit = world_scan(w, 1, 0.5, 10.0)
    assert hit[0, 0] == 2 and fr[0, 0] == f32(0.25)
    assert hit[1, 0] == 2   # agent 1 looks along +x from inside agent 0's disc: it reports agent 2, not 0


def test_equal_fractions_lowest_index_wins():
    for lo_above in (True, False):
        y = 0.3 if lo_above else -0.3
        fr, hit = world_scan(make_world([(0, 0), (3, y), (3, -y)], [0, 0, 0]), 1, 0.5, 10.0)
        f1, _ = world_scan(make_world([(0, 0), (3, y)], [0, 0]), 1, 0.5, 10.0)
        assert hit[0, 0] == 1 and same_bits(fr[0, 0], f1[0, 0])


def test_dead_agent_is_transparent():
    w = make_world([(0, 0), (3, 0), (6, 0)], [0, 0, np.pi], dead=[1])
    fr, hit = world_scan(w, 1, 0.5, 10.0)
    assert hit[0, 0] == 2 and fr[0, 0] == f32(0.55)
    assert hit[1, 0] == 2                 # the dead agent still scans
    assert hit[2, 0] == 0                 # and agent 2 looks back through it to agent 0


def test_middle_ray_points_along_the_heading():
    a = 0.7
    o = 1.0 * ((2 * np.arange(5) + 1 - 5) / 10.0)
    assert o[2] == 0.0 and np.allclose(o, -o[::-1])
    w = make_world([(0, 0), (3 * np.cos(a), 3 * np.sin(a))], [a, 0])
    fr, hit = world_scan(w, 5, 1.0, 10.0)
    assert hit[0].tolist() == [-1, -1, 1, -1, -1]
    assert abs(fr[0, 2] - 0.25) < 1e-6
    # r counts counter-clockwise: a body 1.2 m to the left (half-width asin(0.5 / 1.2) = 24.6 degrees)
    w = make_world([(0, 0), (0, 1.2)], [0, 0])
    _, hit = world_scan(w, 4, 2 * np.pi, 10.0)   # rays at -3pi/4, -pi/4, pi/4, 3pi/4: 45 degrees off, missed
    assert hit[0].tolist() == [-1, -1, -1, -1]
    _, hit = world_scan(w, 8, 2 * np.pi, 10.0)   # rays at -7pi/8 .. 7pi/8 in steps of pi/4: 3pi/8 and 5pi/8 meet it
    assert hit[0].tolist() == [-1, -1, -1, -1, -1, 1, 1, -1]


def test_lidar_args_layout_matches_header():
    from gym_macm import _lib
    hdr = open(os.path.join(ROOT, "include", "macm.h")).read()
    body = hdr[hdr.index("typedef struct macm_lidar_args {"):hdr.index("} macm_lidar_args;")]
    fields = []
    for line in body.splitlines()[1:]:
        m = re.match(r"\s*(?:const\s+)?(int32_t|double|void)(\*?)\s+([^;]+);", line.split("/*")[0])
        if m:
            kind = "ptr" if m.group(2) else m.group(1)
            fields += [(n.strip().lstrip("*"), kind) for n in m.group(3).split(",")]
    ctypes_kind = {_lib.i32: "int32_t", _lib.f64: "double"}
    assert fields == [(n, ctypes_kind.get(t, "ptr")) for n, t in _lib.MacmLidarArgs._fields_]
    assert _lib.MAX_RAYS == int(re.search(r"#define MACM_MAX_RAYS (\d+)", hdr).group(1))
    assert "macm_lidar" in _lib.EXPORTS


def test_python_rejects_bad_arguments_before_the_call():
    from gym_macm import batched
    fake = types.SimpleNamespace()   # fails on any use: the checks come first
    bad = [dict(n_rays=0, max_range=1.0), dict(n_rays=1025, max_range=1.0), dict(n_rays=2.0, max_range=1.0),
           dict(n_rays=True, max_range=1.0), dict(n_rays=8, max_range=0.0), dict(n_rays=8, max_range=-1.0),
           dict(n_rays=8, max_range=math.inf), dict(n_rays=8, max_range=math.nan), dict(n_rays=8, max_range=1e6 + 1),
           dict(n_rays=8, max_range=1.0, fov=0.0), dict(n_rays=8, max_range=1.0, fov=-1.0),
           dict(n_rays=8, max_range=1.0, fov=2 * math.pi + 1e-9), dict(n_rays=8, max_range=1.0, fov=math.nan),
           dict(n_rays=8, max_range=1.0, out=()), dict(n_rays=8, max_range=1.0, out="ab")]
    for kw in bad:
        with pytest.raises(ValueError):
            batched._BatchedCommon.lidar(fake, **kw)
