"""Known answers DERIVED BY HAND FROM THE REFERENCE'S RUST TEXT -- not produced by the oracle.

The reference's own tests pin only transform / AABB / camera arithmetic (tests/test_oracle_kat.py).  For the
outputs of the hot path -- which shape is hit, t, normal, point, (u, v), front face, the scatter direction and
the pixel colour -- the reference holds no golden vector, and the Rust crate cannot be built in this image.
This file closes that gap as far as it can be closed without running the reference: every case below is a
small scene and one ray whose result follows from the cited Rust lines by hand; the derivation is in the
comment next to the expected value.  Each case is checked

  * against the ORACLE (CPU suite): a transcription slip in oracle/oracle.cpp shows up here, and
  * against the CUDA path through the C ABI (`-m gpu`): rt_intersect_batch in both modes (the literal loop
    and cull tree + exact-skip marching) and rt_trace_pixel_samples (= renderer::trace_pixel_samples).

Tolerances (stated per case): values that are exactly representable are compared with `==`; values that
involve pi, a square root or a marched root are compared to 1e-12 / 2e-8 as noted.

Citations are into /root/reference/src (shapes = world/shapes/mod.rs, march = world/shapes/ray_marching.rs).
"""
import json
import math
import os

import numpy as np
import pytest

import rs_pathtracing_b200 as rt
from oracle import pyoracle as po

IDENT = {"translate": [0, 0, 0], "rotate": [0, 0, 0], "scale": [1, 1, 1]}
CAMERA = {"position": [0, 0, -10], "direction": [0, 0, 1], "up": [0, 1, 0], "fov": 40.0, "focal_length": 1.0}
INF = math.inf


def xf(translate=(0, 0, 0), scale=(1, 1, 1), rotate=(0, 0, 0)):
    return {"translate": list(translate), "rotate": list(rotate), "scale": list(scale)}


def solid(c):
    return {"type": "SolidColor", "color": list(c)}


GREY = {"type": "Lambertian", "albedo": solid((0.5, 0.5, 0.5))}


def sphere(transform=IDENT, material="M", **kw):
    return dict({"type": "Sphere", "name": "s", "material": material, "transform": transform}, **kw)


def cube(transform=IDENT, material="M"):
    return {"type": "Cube", "name": "c", "material": material, "transform": transform}


def rect(x0=-1.0, y0=-1.0, x1=1.0, y1=1.0, transform=IDENT, material="M"):
    return {"type": "Rectangle", "x0": x0, "y0": y0, "x1": x1, "y1": y1, "material": material, "transform": transform}


def marched(surface, transform=IDENT, material="M", step=0.01, **kw):
    return dict({"type": "BruteForsableShape", "shape": surface, "step": step, "material": material,
                 "transform": transform}, **kw)


def make_scene(shapes, materials=None):
    text = json.dumps({"camera": CAMERA, "background": [0, 0, 0], "materials": materials or {"M": GREY},
                       "shapes": shapes})
    return rt.Scene.from_json(text, add_random_spheres=False)


def ray(o, d):
    """rt_ray as the kernels take it: the direction is used AS GIVEN (Ray::new normalises, world/ray.rs:12-17;
    every direction below already has unit length, so Ray::new would leave it unchanged)."""
    assert abs(math.sqrt(sum(x * x for x in d)) - 1.0) < 1e-15
    return np.array([list(o) + list(d)], dtype=np.float64)


PI = math.pi

# ------------------------------------------------------------------------------------------------
# (1) nearest hit: index, t, point, normal, (u, v), front face
# ------------------------------------------------------------------------------------------------
# Each case: (id, shapes, ray origin, ray direction, t_min, t_max, expected).  `expected` = None for a miss, else a
# dict with index / t / point / normal / uv / front; "tol" = absolute tolerance on t, point, normal, uv (0 = exact).
HIT_CASES = []


def case(name, shapes, o, d, want, t_min=0.001, t_max=INF):
    HIT_CASES.append(pytest.param(shapes, o, d, t_min, t_max, want, id=name))


# --- Sphere (shapes:330-374) ------------------------------------------------------------------------
# test_torus's ray (shapes:853-860), origin (0,0,-10) direction +z, against the unit Sphere:
#   a = d.d = 1, half_b = d.o = -10, c = o.o - 1 = 99, D = 100 - 99 = 1 > 0
#   x = (-half_b - sqrt(D)) / a = (10 - 1) / 1 = 9, inside [0.001, inf)          -> t = 9
#   p = o + d x = (0, 0, -1); normal = p = (0, 0, -1); n.d = -1 < 0              -> front face, normal kept
#   theta = acos(-p.y) = acos(-0) = pi/2                                          -> v = theta / pi = 0.5
#   phi = atan2(-p.z, p.x) + pi = atan2(1, 0) + pi = 3 pi / 2                     -> u = phi / 2 pi = 0.75
case("sphere_head_on", [sphere()], (0, 0, -10), (0, 0, 1),
     dict(index=0, t=9.0, point=(0, 0, -1), normal=(0, 0, -1), uv=(0.75, 0.5), front=1, tol=1e-15))
# The same sphere translated to z = 5 and scaled by 2 (radius 2 in the world), ray from the origin along +z.
# Shape::ray_hit_transformed (shapes:112-124) intersects in object space with the un-normalised direction
# (transform.rs:32-37): o' = S^-1 (o - T) = (0, 0, -2.5), d' = (0, 0, 0.5):
#   a = 0.25, half_b = -1.25, c = 6.25 - 1 = 5.25, D = 1.5625 - 1.3125 = 0.25, sqrt = 0.5
#   x = (1.25 - 0.5) / 0.25 = 3 (the world distance: the sphere's near pole is at z = 3)
#   p' = (0, 0, -1); point = direct p' = T + S p' = (0, 0, 3); normal = inverse^T p' = (0, 0, -0.5) -> (0, 0, -1)
case("sphere_scaled_translated", [sphere(xf((0, 0, 5), (2, 2, 2)))], (0, 0, 0), (0, 0, 1),
     dict(index=0, t=3.0, point=(0, 0, 3), normal=(0, 0, -1), uv=(0.75, 0.5), front=1, tol=1e-15))
# From the centre of the unit sphere along +x: a = 1, half_b = 0, c = -1, D = 1;
#   near root (0 - 1)/1 = -1 < t_min -> far root (0 + 1)/1 = 1 (shapes:345-352)
#   p = (1, 0, 0); normal = p; n.d = 1 > 0 -> NOT front; set_normal (ray.rs:60-64) flips it to (-1, 0, 0)
#   p.z = 0 + 0*1 = 0, -p.z = -0.0: atan2(-0.0, 1) = -0.0, phi = pi -> u = 0.5; acos(-0.0) = pi/2 -> v = 0.5
case("sphere_from_inside", [sphere()], (0, 0, 0), (1, 0, 0),
     dict(index=0, t=1.0, point=(1, 0, 0), normal=(-1, 0, 0), uv=(0.5, 0.5), front=0, tol=1e-15))
# inverse_normal (shapes:359): normal = -p = (0, 0, 1); n.d = 1 > 0 -> not front, flipped back to (0, 0, -1)
case("sphere_inverse_normal", [sphere(inverse_normal=True)], (0, 0, -10), (0, 0, 1),
     dict(index=0, t=9.0, point=(0, 0, -1), normal=(0, 0, -1), uv=(0.75, 0.5), front=0, tol=1e-15))
# The D == 0 quirk (shapes:343-344): `-half_b * a`, a MULTIPLICATION, and no range check.  Sphere scaled by 2,
# ray o = (2, 0, -4), d = +z touches it: o' = (1, 0, -2), d' = (0, 0, 0.5):
#   a = 0.25, half_b = -1, c = 1 + 4 - 1 = 4, D = 1 - 0.25*4 = 0 exactly
#   x = -half_b * a = 0.25   (the tangent point is really at x = 4)
#   p' = (1, 0, -2 + 0.5*0.25) = (1, 0, -1.875), |p'| = sqrt(1 + 3.515625) = 2.125 exactly
#   point = 2 p' = (2, 0, -3.75); normal = normalize(inverse^T normalize(p')) = p' / 2.125; n.d < 0 -> front
#   v = acos(-0)/pi = 0.5; u = (atan2(1.875, 1) + pi) / 2 pi
_N = (1 / 2.125, 0.0, -1.875 / 2.125)
_U = (math.atan2(1.875, 1.0) + PI) / (2 * PI)
case("sphere_tangent_quirk", [sphere(xf((0, 0, 0), (2, 2, 2)))], (2, 0, -4), (0, 0, 1),
     dict(index=0, t=0.25, point=(2, 0, -3.75), normal=_N, uv=(_U, 0.5), front=1, tol=1e-15))
# ... "accepted without range check": the same hit with max_t = 0.1 < 0.25 and with t_min = 1 > 0.25
case("sphere_tangent_quirk_ignores_max_t", [sphere(xf((0, 0, 0), (2, 2, 2)))], (2, 0, -4), (0, 0, 1),
     dict(index=0, t=0.25, point=(2, 0, -3.75), normal=_N, uv=(_U, 0.5), front=1, tol=1e-15), t_max=0.1)
case("sphere_tangent_quirk_ignores_t_min", [sphere(xf((0, 0, 0), (2, 2, 2)))], (2, 0, -4), (0, 0, 1),
     dict(index=0, t=0.25, point=(2, 0, -3.75), normal=_N, uv=(_U, 0.5), front=1, tol=1e-15), t_min=1.0)
# D < 0: o = (2, 0, -10), d = +z against the unit sphere: c = 103, D = 100 - 103 < 0 -> None (shapes:341-342)
case("sphere_miss", [sphere()], (2, 0, -10), (0, 0, 1), None)
# both roots beyond max_t / behind the origin -> None (shapes:346-351)
case("sphere_beyond_max_t", [sphere()], (0, 0, -10), (0, 0, 1), None, t_max=8.0)
case("sphere_behind", [sphere()], (0, 0, 10), (0, 0, 1), None)

# --- Cube (shapes:250-285) ---------------------------------------------------------------------------
# o = (0.25, -0.5, -5), d = +z against the unit box [-1, 1]^3:
#   t_lower = (-1 - o) / d = (-1.25/0, -0.5/0, 4/1) = (-inf, -inf, 4); t_upper = (0.75/0, 1.5/0, 6/1) = (inf, inf, 6)
#   t_box_min = max(max(-inf, -inf, 4), 0.001) = 4; t_box_max = min(min(inf, inf, 6), inf) = 6    -> t = 4
#   p = o + 4 d = (0.25, -0.5, -1); |p| = (0.25, 0.5, 1), max = |p.z| -> normal (0, 0, p.z) = (0, 0, -1), (u, v) = (p.x, p.y)
case("cube_face", [cube()], (0.25, -0.5, -5), (0, 0, 1),
     dict(index=0, t=4.0, point=(0.25, -0.5, -1), normal=(0, 0, -1), uv=(0.25, -0.5), front=1, tol=0))
# origin INSIDE the box (shapes:257-263): o = 0, d = +x: t_lower = (-1, -inf, -inf), t_upper = (1, inf, inf)
#   t_box_min = max(max(-1, -inf, -inf), t_min) = t_min = 0.001 -- the hit is reported AT t_min, not at the exit
#   p = (0.001, 0, 0); max |p| = |p.x| -> normal (0.001, 0, 0) -> (1, 0, 0); n.d > 0 -> not front, flipped; (u, v) = (p.y, p.z)
case("cube_from_inside_hits_at_t_min", [cube()], (0, 0, 0), (1, 0, 0),
     dict(index=0, t=0.001, point=(0.001, 0, 0), normal=(-1, 0, 0), uv=(0, 0), front=0, tol=0))
# Cube translated to z = 10, scaled (1, 1, 2): world box z in [8, 12].  o' = (0, 0, -5), d' = (0, 0, 0.5):
#   t_lower.z = (-1 + 5)/0.5 = 8, t_upper.z = 12 -> t = 8; p' = (0, 0, -1); point = T + S p' = (0, 0, 8)
#   normal = inverse^T (0, 0, -1) = (0, 0, -0.5) -> (0, 0, -1)
case("cube_scaled_translated", [cube(xf((0, 0, 10), (1, 1, 2)))], (0, 0, 0), (0, 0, 1),
     dict(index=0, t=8.0, point=(0, 0, 8), normal=(0, 0, -1), uv=(0, 0), front=1, tol=0))
# slab miss: o = (3, 0, -5), d = +z: t_lower.x = -4/0 = -inf, t_upper.x = -2/0 = -inf -> t_box_max = -inf < t_box_min
case("cube_miss", [cube()], (3, 0, -5), (0, 0, 1), None)

# --- Rectangle (shapes:181-204) ----------------------------------------------------------------------
# z = 0 plane clipped to [-1, 1]^2; o = (0.25, 0.5, -3), d = +z: t = -o.z/d.z = 3; p = (0.25, 0.5, 0) inside
#   u = (0.25 + 1)/2 = 0.625, v = (0.5 + 1)/2 = 0.75; normal (0, 0, 1); n.d = 1 > 0 -> not front, flipped to (0, 0, -1)
case("rect_hit", [rect()], (0.25, 0.5, -3), (0, 0, 1),
     dict(index=0, t=3.0, point=(0.25, 0.5, 0), normal=(0, 0, -1), uv=(0.625, 0.75), front=0, tol=0))
# from the other side: o = (0.25, 0.5, 3), d = -z: t = -3 / -1 = 3; n.d = -1 < 0 -> front, normal stays (0, 0, 1)
case("rect_hit_front", [rect()], (0.25, 0.5, 3), (0, 0, -1),
     dict(index=0, t=3.0, point=(0.25, 0.5, 0), normal=(0, 0, 1), uv=(0.625, 0.75), front=1, tol=0))
# p.x = 1.5 > x1 -> None; and a hit exactly ON the edge x = x1 is inside (`p.x > self.x1` is false, shapes:187)
case("rect_outside", [rect()], (1.5, 0, -3), (0, 0, 1), None)
case("rect_edge_inclusive", [rect()], (1.0, 0, -3), (0, 0, 1),
     dict(index=0, t=3.0, point=(1, 0, 0), normal=(0, 0, -1), uv=(1.0, 0.5), front=0, tol=0))
# a ray lying IN the plane: t = -0/0 = NaN; `t < min_t || t > max_t` is false for NaN, p = o + d NaN = NaN, the four
# bounds comparisons are false as well -> Some(hit) with t = NaN (SURVEY A.6)
case("rect_in_plane_nan", [rect()], (0, 0, 0), (1, 0, 0), dict(index=0, t=math.nan, front=None, tol=0))

# --- ShapeCollection (shapes:573-597) -----------------------------------------------------------------
# two coincident unit spheres: the loop calls ray_hit(ray, min_t, min_distance) and every shape accepts
# t == max_t (`x > max_t` rejects, shapes:347), so the LATER shape replaces the earlier one on a tie
case("collection_tie_later_wins", [sphere(), sphere()], (0, 0, -10), (0, 0, 1),
     dict(index=1, t=9.0, point=(0, 0, -1), normal=(0, 0, -1), uv=(0.75, 0.5), front=1, tol=1e-15))
# a sphere of radius 0.5 at z = -3 in front of the unit cube: sphere t = 10 - 3 - 0.5 = 6.5 < cube t = 9, in either order
case("collection_nearest_first", [sphere(xf((0, 0, -3), (0.5, 0.5, 0.5))), cube()], (0, 0, -10), (0, 0, 1),
     dict(index=0, t=6.5, point=(0, 0, -3.5), normal=(0, 0, -1), uv=(0.75, 0.5), front=1, tol=1e-15))
case("collection_nearest_last", [cube(), sphere(xf((0, 0, -3), (0.5, 0.5, 0.5)))], (0, 0, -10), (0, 0, 1),
     dict(index=1, t=6.5, point=(0, 0, -3.5), normal=(0, 0, -1), uv=(0.75, 0.5), front=1, tol=1e-15))


# --- RayMarchingShape (march:20-74) --------------------------------------------------------------------
# The six surface functions and gradients, transcribed here from the Rust text independently of the oracle
# (march:147-168, 203-237, 268-300, 340-369, 399-434, 464-504).
def f_heart(x, y, z):
    x2, y2, z2 = x * x, y * y, z * z
    z3 = z2 * z
    a = x2 + (9.0 / 4.0) * y2 + z2 - 1.0
    return a * a * a - x2 * z3 - (9.0 / 80.0) * y2 * z3


def g_heart(x, y, z):
    a = x * x + (9.0 / 4.0) * y * y + z * z - 1.0
    a = 3.0 * a * a
    z2 = z * z
    z3 = z2 * z
    return (2.0 * x * (a - z3), (9.0 / 2.0) * y * (a - 0.05 * z3), 2.0 * z * (a - z * (1.5 * x * x + (27.0 / 40.0) * y * y)))


def f_sine(x, y, z, a):
    return a * a * (x - y - z) * (x + y - z) * (x - y + z) * (x + y + z) + 4.0 * x * x * y * y * z * z


def g_sine(x, y, z, a):
    x2, y2, z2, a2 = x * x, y * y, z * z, a * a
    return (4.0 * x * (a2 * (x2 - y2 - z2) + 2.0 * y2 * z2), 8.0 * x2 * y * z2 - 4.0 * a2 * y * (x2 - y2 + z2),
            8.0 * x2 * y2 * z - 4.0 * a2 * z * (x2 + y2 - z2))


def f_star(x, y, z, a):
    x2, y2, z2 = x * x, y * y, z * z
    c = x2 + y2 + z2 - 1.0
    return a * (x2 * y2 + x2 * z2 + y2 * z2) + (c * c * c)


def g_star(x, y, z, a):
    x2, y2, z2 = x * x, y * y, z * z
    c = x2 + y2 + z2 - 1.0
    return (2.0 * a * x * (y2 + z2) + 6.0 * x * c * c, 2.0 * a * y * (x2 + z2) + 6.0 * y * c * c,
            2.0 * a * z * (x2 + y2) + 6.0 * z * c * c)


def f_dupin(x, y, z, a, b, c, d):
    b2 = b * b
    e = x * x + y * y + z * z + b2 - d * d
    f = a * x - c * d
    return e * e - 4.0 * (f * f + b2 * y * y)


def g_dupin(x, y, z, a, b, c, d):
    b2 = b * b
    e = 4.0 * (x * x + y * y + z * z + b2 - d * d)
    return (e * x - 8.0 * a * (a * x - c * d), e * y - 8.0 * b2 * y, e * z)


def f_hunts(x, y, z):
    x2, y2, z2 = x * x, y * y, z * z
    a = x2 + y2 + z2 - 13.0
    b = 3.0 * x2 + y2 - 4.0 * z2 - 12.0
    return 4.0 * a * a * a + 27.0 * b * b


def g_hunts(x, y, z):
    x2, y2, z2 = x * x, y * y, z * z
    a = x2 + y2 + z2 - 13.0
    b = 3.0 * x2 + y2 - 4.0 * (z2 + 3.0)
    return (24.0 * x * a * a + 324.0 * x * b, 12.0 * y * (2.0 * a * a + 9.0 * b), 24.0 * z * (a * a - 18.0 * b))


def f_cushion(x, y, z):
    x2, y2, z2 = x * x, y * y, z * z
    a = x2 - z
    return (z2 * x2 - z2 * z2 - 2.0 * z * x2 + 2.0 * z * z2 + x2 - z2 - a * a - y2 * y2 - 2.0 * x2 * y2 - y2 * z2
            + 2.0 * y2 * z + y2)


def g_cushion(x, y, z):
    x2, y2, z2 = x * x, y * y, z * z
    return (2.0 * x * (-2.0 * x2 - 2.0 * y2 + z2 + 1.0), -2.0 * y * (2.0 * x2 + 2.0 * y2 + z2 - 2.0 * z - 1.0),
            2.0 * z * (x2 - 2.0 * z2 + 3.0 * z - 2.0) - 2.0 * y * (z - 1.0))


# (JSON description, f, gradient, params8 of the flat scene: [kind, step, depth, a, b, c, d, sphere_radius], uv rule)
SURFACES = {
    "Heart": ({"type": "Heart"}, f_heart, g_heart, (), False),
    "Sine": ({"type": "Sine", "a": 0.8, "sphere_radius": 2.0}, lambda x, y, z: f_sine(x, y, z, 0.8),
             lambda x, y, z: g_sine(x, y, z, 0.8), (0.8,), False),
    "Star": ({"type": "Star", "a": 50.0, "sphere_radius": 1.5}, lambda x, y, z: f_star(x, y, z, 50.0),
             lambda x, y, z: g_star(x, y, z, 50.0), (50.0,), False),
    "DupinCyclide": ({"type": "DupinCyclide", "a": 1.11, "b": 0.99, "c": 0.5, "d": 0.1, "sphere_radius": 2.5},
                     lambda x, y, z: f_dupin(x, y, z, 1.11, 0.99, 0.5, 0.1),
                     lambda x, y, z: g_dupin(x, y, z, 1.11, 0.99, 0.5, 0.1), (1.11, 0.99, 0.5, 0.1), True),
    "HuntsSurface": ({"type": "HuntsSurface", "sphere_radius": 4.5}, f_hunts, g_hunts, (), True),
    "Cushion": ({"type": "Cushion", "sphere_radius": 1.5}, f_cushion, g_cushion, (), True),
}


def first_root(f, o, d, start, end, step=0.01):
    """The root the reference's loop brackets: walk t = start, start + step, ... until f changes sign (march:27-49),
    then bisect that bracket in plain Python.  Independent of the oracle; precision ~1e-15."""
    fx = lambda t: f(o[0] + t * d[0], o[1] + t * d[1], o[2] + t * d[2])
    t, r = start, fx(start)
    while t <= end:
        nt = t + step
        nx = fx(nt)
        if (r < 0 < nx) or (r > 0 > nx):
            lo, hi = t, nt
            for _ in range(200):
                mid = 0.5 * (lo + hi)
                if (fx(mid) < 0) == (r < 0):
                    lo = mid
                else:
                    hi = mid
            return 0.5 * (lo + hi)
        t, r = nt, nx
    return None


def sphere_bound(o, d, radii):
    """intersect_bound (march:135-145 Heart, :213-225 the others): roots of |(o + t d) / radii| = 1, clamped at 0"""
    oo = [o[k] / radii[k] for k in range(3)]
    dd = [d[k] / radii[k] for k in range(3)]
    a = sum(x * x for x in dd)
    hb = sum(x * y for x, y in zip(dd, oo))
    c = sum(x * x for x in oo) - 1.0
    disc = hb * hb - a * c
    assert disc > 0
    return max((-hb - math.sqrt(disc)) / a, 0.0), max((-hb + math.sqrt(disc)) / a, 0.0)


def marched_case(name, key, o, d, scale=1.0, translate=(0, 0, 0)):
    """March:20-74 for a surface under translate + uniform scale.  The loop walks t in steps of 0.01 from the bound's
    entry, reverses with step *= -0.01 at each sign change, four times (depth 4): after the fourth bracket the
    sample sits within the last step (0.01 * 0.01^3 = 1e-8) of the root it has been closing in on, so
        |t - t_root| <= 1e-8  (+ accumulated rounding, < 1e-12)            -> tolerance 2e-8
    unless |f| < 1e-15 ends the search earlier at a sample even closer to the root.  The ray is transformed to
    object space WITHOUT renormalising (transform.rs:32-37), so t is the world distance; the point returned is
    direct * p', the normal inverse^T * gradient(p') face-forwarded and normalised; (u, v) = (p'.x, p'.y) for
    Dupin / Hunt / Cushion and (0, 0) for Heart / Sine / Star (march:59-61 and the uv() impls)."""
    js, f, g, _, uv_xy = SURFACES[key]
    oo = [(o[k] - translate[k]) / scale for k in range(3)]
    dd = [d[k] / scale for k in range(3)]
    radii = (1.45, 1.45 / 2.05, 1.45) if key == "Heart" else (js["sphere_radius"],) * 3
    start, end = sphere_bound(oo, dd, radii)
    t = first_root(f, oo, dd, start, end)
    assert t is not None, name
    p = [oo[k] + t * dd[k] for k in range(3)]
    n = [x / scale for x in g(*p)]               # inverse^T of a uniform scale
    if sum(n[k] * d[k] for k in range(3)) > 0:   # set_normal: oppose the ray
        n, front = [-x for x in n], 0
    else:
        front = 1
    ln = math.sqrt(sum(x * x for x in n))
    want = dict(index=0, t=t, point=tuple(translate[k] + scale * p[k] for k in range(3)),
                normal=tuple(x / ln for x in n), uv=(p[0], p[1]) if uv_xy else (0.0, 0.0), front=front, tol=2e-8,
                tol_point=2e-8 * max(1.0, scale), tol_normal=1e-5)
    case(name, [marched(js, xf(translate, (scale,) * 3))], o, d, want)


marched_case("march_heart", "Heart", (0.3, 0.2, -3.0), (0.0, 0.0, 1.0))
marched_case("march_heart_scaled_10", "Heart", (3.0, 2.0, -30.0), (0.0, 0.0, 1.0), scale=10.0)
marched_case("march_heart_cornell_scale", "Heart", (278.0 + 20.0, 200.0 + 10.0, -800.0), (0.0, 0.0, 1.0), scale=82.5,
             translate=(278.0, 200.0, 278.0))
marched_case("march_sine", "Sine", (0.4, 0.3, -3.0), (0.0, 0.0, 1.0))
marched_case("march_star", "Star", (0.35, 0.2, -3.0), (0.0, 0.0, 1.0))
marched_case("march_dupin", "DupinCyclide", (1.0, 0.2, -4.0), (0.0, 0.0, 1.0))
marched_case("march_dupin_along_x", "DupinCyclide", (-4.0, 0.2, 0.3), (1.0, 0.0, 0.0))
marched_case("march_hunts", "HuntsSurface", (0.5, 0.3, -6.0), (0.0, 0.0, 1.0))
marched_case("march_cushion", "Cushion", (0.2, 0.1, -3.0), (0.0, 0.0, 1.0))
# through the Heart's bounding ellipsoid but past the surface: x = 1.3 > every point of the heart (|x| < 1.2):
# the loop runs until t > end -> None (march:29-31)
case("march_heart_bound_only", [marched({"type": "Heart"})], (1.3, 0.0, -3.0), (0.0, 0.0, 1.0), None)
# through the hole of the cyclide: f keeps its sign along the whole chord (checked by first_root at import)
assert first_root(SURFACES["DupinCyclide"][1], (0.3, 0.2, -4.0), (0.0, 0.0, 1.0),
                  *sphere_bound((0.3, 0.2, -4.0), (0.0, 0.0, 1.0), (2.5, 2.5, 2.5))) is None
case("march_dupin_through_the_hole", [marched(SURFACES["DupinCyclide"][0])], (0.3, 0.2, -4.0), (0.0, 0.0, 1.0), None)


def _check_hit(got, want, label):
    if want is None:
        assert got["index"][0] == -1, f"{label}: expected a miss, got shape {got['index'][0]}"
        return
    assert got["index"][0] == want["index"], f"{label}: index {got['index'][0]} != {want['index']}"
    tol = want["tol"]
    if math.isnan(want["t"]):
        assert math.isnan(got["t"][0]), label
        return
    assert abs(got["t"][0] - want["t"]) <= tol, f"{label}: t {got['t'][0]!r} != {want['t']!r}"
    assert np.abs(got["point"][0] - np.array(want["point"], float)).max() <= want.get("tol_point", tol), \
        f"{label}: point {got['point'][0]} != {want['point']}"
    assert np.abs(got["normal"][0] - np.array(want["normal"], float)).max() <= want.get("tol_normal", tol), \
        f"{label}: normal {got['normal'][0]} != {want['normal']}"
    assert np.abs(got["uv"][0] - np.array(want["uv"], float)).max() <= max(tol, 1e-15), \
        f"{label}: uv {got['uv'][0]} != {want['uv']}"
    assert got["front"][0] == want["front"], f"{label}: front face {got['front'][0]} != {want['front']}"


@pytest.mark.parametrize("shapes,o,d,t_min,t_max,want", HIT_CASES)
def test_oracle_reproduces_the_source_derived_hits(shapes, o, d, t_min, t_max, want):
    sc = make_scene(shapes)
    got = po.OracleScene(sc.desc()).intersect_batch(ray(o, d), t_min, t_max)
    _check_hit(got, want, "oracle")


@pytest.mark.gpu
@pytest.mark.parametrize("shapes,o,d,t_min,t_max,want", HIT_CASES)
def test_cuda_reproduces_the_source_derived_hits(shapes, o, d, t_min, t_max, want):
    sc = make_scene(shapes)
    for mode in (rt.RT_ISECT_BRUTE, rt.RT_ISECT_FAST):
        _check_hit(sc.closest_hit(ray(o, d), t_min, t_max, mode=mode), want, f"cuda mode {mode}")


def test_oracle_surface_functions_match_the_independent_transcription():
    """oracle/oracle.cpp's six polynomials and gradients against the transcriptions above, at random points:
    same operand order, so the same bits (the gradients keep the reference's own quirks, e.g. Heart's 27/40)."""
    rng = np.random.default_rng(5)
    kinds = {"Heart": 0, "Sine": 1, "Star": 2, "DupinCyclide": 3, "HuntsSurface": 4, "Cushion": 5}
    import ctypes as C
    for key, (js, f, g, abcd, _) in SURFACES.items():
        params = np.zeros(8)
        params[0] = kinds[key]
        params[1], params[2] = 0.01, 4
        params[3:3 + len(abcd)] = abcd
        params[7] = js.get("sphere_radius", 0.0)
        pp = params.ctypes.data_as(C.POINTER(C.c_double))
        for p in rng.uniform(-2.0, 2.0, (64, 3)):
            assert po.lib().orc_surface_func(pp, po.Vec3(*p)) == f(*p), key
            assert po.lib().orc_surface_gradient(pp, po.Vec3(*p)).tuple() == tuple(g(*p)), key


# ------------------------------------------------------------------------------------------------
# (2) materials, textures, ray_color: one path per case through trace_pixel_samples
# ------------------------------------------------------------------------------------------------
SKY_Z = (0.75, 0.85, 1.0)   # Scene::background (world/mod.rs:199-202) for dir.y = 0: t = 0.5 -> 0.5 (1,1,1) + 0.5 (0.5,0.7,1)
SEED, PIXEL = 11, 5


def sky(d):
    t = 0.5 * (d[1] + 1.0)
    return tuple((1.0 - t) * 1.0 + t * c for c in (0.5, 0.7, 1.0))


def draws(event, n, sample=0):
    """the generator's stream for (seed, pixel, sample, event): the values `rng.gen()` returns, in order
    (tests/test_oracle_kat.py pins the Philox rounds against Random123's known answers)"""
    return po.philox_stream(SEED, PIXEL, sample, event, n)


def random_in_unit_sphere(u):
    """algebra/mod.rs:59-84: Vector3d::random(-1, 1) = three gen_range draws, retried until |v|^2 <= 1"""
    for k in range(0, len(u) - 2, 3):
        v = [-1.0 + 2.0 * u[k + j] for j in range(3)]
        if v[0] * v[0] + v[1] * v[1] + v[2] * v[2] <= 1.0:
            return v
    raise AssertionError("no accepted sample in the draws provided")


def normalize(v):
    ln = math.sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2])
    return [x / ln for x in v]


COLOR_CASES = []


def color_case(name, shapes, materials, o, d, depth, want, tol=1e-12):
    COLOR_CASES.append(pytest.param(shapes, materials, o, d, depth, want, tol, id=name))


ALBEDO = (0.8, 0.4, 0.2)
# miss -> Scene::background: straight up t = 1 -> (0.5, 0.7, 1.0); straight down t = 0 -> (1, 1, 1); horizontal -> SKY_Z
color_case("sky_up", [sphere(xf((50, 0, 0)))], None, (0, 0, 0), (0, 1, 0), 8, (0.5, 0.7, 1.0), tol=0)
color_case("sky_down", [sphere(xf((50, 0, 0)))], None, (0, 0, 0), (0, -1, 0), 8, (1.0, 1.0, 1.0), tol=0)
color_case("sky_horizontal", [sphere(xf((50, 0, 0)))], None, (0, 0, 0), (0, 0, 1), 8, SKY_Z, tol=0)
# ray_color with depth == 0: any hit is black (renderer/mod.rs:26-27) -- also an emitter
LIGHT = {"type": "DiffuseLight", "emit": solid((15, 15, 15))}
color_case("depth_0_is_black", [sphere()], {"M": GREY}, (0, 0, -10), (0, 0, 1), 0, (0, 0, 0), tol=0)
color_case("depth_0_emitter_is_black", [sphere()], {"M": LIGHT}, (0, 0, -10), (0, 0, 1), 0, (0, 0, 0), tol=0)
# DiffuseLight: scatter = None -> emitted(u, v, p) = the texture's colour (material.rs:123-127, renderer/mod.rs:34-36)
color_case("emitter", [sphere()], {"M": LIGHT}, (0, 0, -10), (0, 0, 1), 8, (15, 15, 15), tol=0)
# EmptyMaterial: scatter None, emitted black (material.rs:130-134)
color_case("empty_material", [sphere()], {"M": {"type": "EmptyMaterial"}}, (0, 0, -10), (0, 0, 1), 8, (0, 0, 0), tol=0)
# Metal, fuzz 0 (material.rs:64-75), head on: hit p = (0,0,-1), n = (0,0,-1); reflect (algebra/mod.rs:122-125) =
# d - 2 (d.n) n = (0,0,1) - 2(-1)(0,0,-1) = (0,0,-1); the reflected ray misses everything -> albedo (x) sky(dir.y = 0)
MIRROR = {"type": "Metal", "albedo": solid(ALBEDO), "fuzz": 0.0}
color_case("metal_mirror_head_on", [sphere()], {"M": MIRROR}, (0, 0, -10), (0, 0, 1), 8,
           tuple(a * s for a, s in zip(ALBEDO, SKY_Z)), tol=0)
# ... with depth 1 the recursion ends in the sky just the same (the miss is tested before depth, renderer/mod.rs:24-43)
color_case("metal_mirror_depth_1", [sphere()], {"M": MIRROR}, (0, 0, -10), (0, 0, 1), 1,
           tuple(a * s for a, s in zip(ALBEDO, SKY_Z)), tol=0)
# Metal mirror hit at 45 degrees: o = (0, s, -10), s = sqrt(1/2), d = +z hits the unit sphere at p = (0, s, -s)
# (a = 1, half_b = -10, c = s^2 + 100 - 1, D = 1 - s^2 = 1/2, x = 10 - s); n = p; reflect = d - 2(-s)(0, s, -s) =
# (0, 2 s^2, 1 - 2 s^2) = (0, 1, 0) up to rounding -> sky straight up (0.5, 0.7, 1.0)
_S = math.sqrt(0.5)
color_case("metal_mirror_45_degrees", [sphere()], {"M": MIRROR}, (0, _S, -10), (0, 0, 1), 8,
           tuple(a * s for a, s in zip(ALBEDO, (0.5, 0.7, 1.0))), tol=1e-12)
# two mirrors facing each other never let the path out: Rectangles at z = +-1 (normals face-forwarded), ray along z
# from between them: every level hits and scatters, at depth 0 the product ends in black (renderer/mod.rs:26-27)
color_case("mirror_corridor_runs_out_of_depth", [rect(transform=xf((0, 0, 1))), rect(transform=xf((0, 0, -1)))],
           {"M": MIRROR}, (0, 0, 0), (0, 0, 1), 8, (0, 0, 0), tol=0)
# emission is NOT added on scattering surfaces: mirror -> emitter.  Rectangle mirror at z = 1 (hit at t = 1), the
# reflected ray (0,0,-1) hits the emitter sphere at z = -5 -> attenuation (x) emitted = albedo * 15
color_case("mirror_then_emitter", [rect(transform=xf((0, 0, 1))), sphere(xf((0, 0, -5)), material="L")],
           {"M": MIRROR, "L": LIGHT}, (0, 0, 0), (0, 0, 1), 8, tuple(15 * a for a in ALBEDO), tol=1e-12)
# ... and an emitter reached at the last level is black: depth 1 -> the emitter is hit with depth == 0
color_case("mirror_then_emitter_out_of_depth", [rect(transform=xf((0, 0, 1))), sphere(xf((0, 0, -5)), material="L")],
           {"M": MIRROR, "L": LIGHT}, (0, 0, 0), (0, 0, 1), 1, (0, 0, 0), tol=0)

# --- textures (texture.rs:17-116) through a mirror Rectangle at z = 1 (reflected ray -> SKY_Z) ----------
ODD, EVEN = (0.1, 0.2, 0.8), (0.9, 0.2, 0.1)


def checker(m):
    return {"type": "Metal", "fuzz": 0.0,
            "albedo": {"type": "CheckerTexture", "odd": solid(ODD), "even": solid(EVEN), "multipliers": list(m)}}


def uv_checker(m):
    return {"type": "Metal", "fuzz": 0.0,
            "albedo": {"type": "UVChecker", "odd": solid(ODD), "even": solid(EVEN), "multipliers": list(m)}}


def times_sky(c):
    return tuple(a * s for a, s in zip(c, SKY_Z))


# CheckerTexture (texture.rs:40-51) uses the WORLD hit point: p = (+-0.25, 0.5, 1), multipliers (1, 1, 1):
# sin(0.25) sin(0.5) sin(1) > 0 -> even; sin(-0.25) sin(0.5) sin(1) < 0 -> odd
color_case("checker_even", [rect(transform=xf((0, 0, 1)))], {"M": checker((1, 1, 1))}, (0.25, 0.5, -3), (0, 0, 1), 8,
           times_sky(EVEN), tol=1e-15)
color_case("checker_odd", [rect(transform=xf((0, 0, 1)))], {"M": checker((1, 1, 1))}, (-0.25, 0.5, -3), (0, 0, 1), 8,
           times_sky(ODD), tol=1e-15)
# a product of exactly 0 is NOT < 0 -> even: p = (0, 0.5, 1), sin(0) = 0
color_case("checker_zero_is_even", [rect(transform=xf((0, 0, 1)))], {"M": checker((1, 1, 1))}, (0.0, 0.5, -3), (0, 0, 1), 8,
           times_sky(EVEN), tol=1e-15)
# UVChecker (texture.rs:78-88): sines = sin(v m0 pi) sin(u m1 pi) -- v pairs with multipliers.0.  Hit (u, v) =
# (0.625, 0.75): multipliers (2, 2): sin(1.5 pi) sin(1.25 pi) = (-1)(-0.707) > 0 -> even;
# multipliers (2, 1): sin(1.5 pi) sin(0.625 pi) = (-1)(+0.924) < 0 -> odd; (1, 2): sin(0.75 pi) sin(1.25 pi) < 0 -> odd
# (swapping u and v would give even for (1, 2)... no: sin(0.625 pi) sin(1.5 pi) < 0 as well; (2, 1) swapped:
# sin(1.25 pi) sin(0.75 pi) < 0 -- so (2, 2) and the pair below at (u, v) = (0.625, 0.25) tell the pairing apart)
color_case("uv_checker_even", [rect(transform=xf((0, 0, 1)))], {"M": uv_checker((2, 2))}, (0.25, 0.5, -3), (0, 0, 1), 8,
           times_sky(EVEN), tol=1e-15)
color_case("uv_checker_odd", [rect(transform=xf((0, 0, 1)))], {"M": uv_checker((2, 1))}, (0.25, 0.5, -3), (0, 0, 1), 8,
           times_sky(ODD), tol=1e-15)
# (u, v) = (0.625, 0.25), multipliers (4, 1): sin(v 4 pi) sin(u pi) = sin(pi) sin(0.625 pi) ~ 1.2e-16 * 0.92 > 0 -> even,
# whereas the swapped pairing sin(u 4 pi) sin(v pi) = sin(2.5 pi) sin(0.25 pi) > 0 as well; use multipliers (3, 1):
# sin(0.75 pi) sin(0.625 pi) > 0 -> even; swapped: sin(1.875 pi) sin(0.25 pi) < 0 -> odd.  The reference's pairing -> EVEN
color_case("uv_checker_v_pairs_with_first_multiplier", [rect(transform=xf((0, 0, 1)))], {"M": uv_checker((3, 1))},
           (0.25, -0.5, -3), (0, 0, 1), 8, times_sky(EVEN), tol=1e-15)


# --- Lambertian and Dielectric need the generator's draws ---------------------------------------------
def lambertian_expected():
    """material.rs:42-53 at the head-on hit p = (0,0,-1), n = (0,0,-1) of the unit sphere: direction = n +
    random_unit() (= normalize(random_in_unit_sphere()), algebra/mod.rs:77-88), Ray::new normalises it; the draws
    are event 1 of the path's stream (the scatter at bounce level 0).  The scattered ray leaves the convex sphere
    (dir.n >= 0) and the scene holds nothing else -> albedo (x) sky(dir)."""
    unit = normalize(random_in_unit_sphere(draws(1, 96)))
    direction = [0.0 + unit[0], 0.0 + unit[1], -1.0 + unit[2]]
    assert max(abs(x) for x in direction) > 1e-3          # (is_zero fallback not in play)
    direction = normalize(direction)
    assert direction[2] < -0.05                           # clearly leaving the sphere
    return tuple(a * s for a, s in zip(ALBEDO, sky(direction)))


def dielectric_expected():
    """material.rs:93-115, ray through the centre of a glass sphere (ior 1.5):
    entry: front face -> ratio = 1/1.5; cos = (-d).n = 1, sin = 0; reflectance(1, ratio) = r0 =
    ((1 - ratio)/(1 + ratio))^2 = (1/5)^2 = 0.04 (:84-88, (1 - cos)^5 = 0); refract when the draw (event 1) >= r0:
    refract (algebra/mod.rs:127-133) = ratio (d + cos n) - sqrt(|1 - 0|) n = 0 - n = d -> straight on;
    exit at t = 2: p = (0,0,1), outward normal flipped to (0,0,-1), not front -> ratio = 1.5, cos = 1, r0 = 0.04
    again, draw of event 2 -> straight on; then the sky at dir.y = 0; attenuation (1,1,1) twice."""
    assert draws(1, 1)[0] > 0.05 and draws(2, 1)[0] > 0.05, "pick another SEED/PIXEL: this one reflects"
    return SKY_Z


@pytest.mark.parametrize("shapes,materials,o,d,depth,want,tol", COLOR_CASES)
def test_oracle_reproduces_the_source_derived_colours(shapes, materials, o, d, depth, want, tol):
    sc = make_scene(shapes, materials)
    got = po.OracleScene(sc.desc()).trace_pixel_samples(ray(o, d), depth, seed=SEED, pixel_index=PIXEL)
    assert np.abs(got - np.array(want, float)).max() <= tol, (got, want)


def assert_float_path(got, want, tol=0.0):
    """a GPU colour of one ray: the oracle's FP64 colour rounded to float once, and off by at most one float ulp.  want is
    that colour derived by hand, within its own f64 tol; f32 rounding is monotone, so the GPU value must be a float in
    [prev(f32(want - tol)), next(f32(want + tol))]"""
    got = np.asarray(got, dtype=np.float64)
    want = np.asarray(want, dtype=np.float64)
    assert np.array_equal(got.astype(np.float32).astype(np.float64), got), (got, want)
    lo = np.nextafter((want - tol).astype(np.float32), np.float32(-np.inf)).astype(np.float64)
    hi = np.nextafter((want + tol).astype(np.float32), np.float32(np.inf)).astype(np.float64)
    assert ((lo <= got) & (got <= hi)).all(), (got.tolist(), want.tolist(), lo.tolist(), hi.tolist())


@pytest.mark.gpu
@pytest.mark.parametrize("shapes,materials,o,d,depth,want,tol", COLOR_CASES)
def test_cuda_reproduces_the_source_derived_colours(shapes, materials, o, d, depth, want, tol):
    sc = make_scene(shapes, materials)
    got = sc.trace_pixel_samples(ray(o, d), depth, seed=SEED, pixel_index=PIXEL)
    # the device keeps a finished path's radiance as float32 (DESIGN 3)
    assert_float_path(got, want, tol)


LAMBERT = {"type": "Lambertian", "albedo": solid(ALBEDO)}
GLASS = {"type": "Dielectric", "index_of_refraction": 1.5}


def _draw_cases():
    return [("lambertian", [sphere()], {"M": LAMBERT}, lambertian_expected()),
            ("dielectric", [sphere()], {"M": GLASS}, dielectric_expected())]


def test_oracle_scatter_follows_the_draws():
    for name, shapes, mats, want in _draw_cases():
        sc = make_scene(shapes, mats)
        got = po.OracleScene(sc.desc()).trace_pixel_samples(ray((0, 0, -10), (0, 0, 1)), 8, seed=SEED, pixel_index=PIXEL)
        assert np.abs(got - np.array(want)).max() <= 1e-12, (name, got, want)


@pytest.mark.gpu
def test_cuda_scatter_follows_the_draws():
    for name, shapes, mats, want in _draw_cases():
        sc = make_scene(shapes, mats)
        got = sc.trace_pixel_samples(ray((0, 0, -10), (0, 0, 1)), 8, seed=SEED, pixel_index=PIXEL)
        assert_float_path(got, want, 1e-12)


def test_oracle_metal_fuzz_follows_the_draws():
    """Metal with fuzz (material.rs:64-75): reflected + fuzz * random_in_unit_sphere(), NOT normalised before the
    scaling, no absorption test.  Head-on hit: reflected = (0,0,-1)."""
    fuzz = 0.5
    v = random_in_unit_sphere(draws(1, 96))
    direction = normalize([fuzz * v[0], fuzz * v[1], -1.0 + fuzz * v[2]])
    want = tuple(a * s for a, s in zip(ALBEDO, sky(direction)))
    sc = make_scene([sphere()], {"M": {"type": "Metal", "albedo": solid(ALBEDO), "fuzz": fuzz}})
    got = po.OracleScene(sc.desc()).trace_pixel_samples(ray((0, 0, -10), (0, 0, 1)), 8, seed=SEED, pixel_index=PIXEL)
    assert np.abs(got - np.array(want)).max() <= 1e-12, (got, want)


@pytest.mark.gpu
def test_cuda_metal_fuzz_follows_the_draws():
    fuzz = 0.5
    v = random_in_unit_sphere(draws(1, 96))
    direction = normalize([fuzz * v[0], fuzz * v[1], -1.0 + fuzz * v[2]])
    want = tuple(a * s for a, s in zip(ALBEDO, sky(direction)))
    sc = make_scene([sphere()], {"M": {"type": "Metal", "albedo": solid(ALBEDO), "fuzz": fuzz}})
    got = sc.trace_pixel_samples(ray((0, 0, -10), (0, 0, 1)), 8, seed=SEED, pixel_index=PIXEL)
    assert_float_path(got, want, 1e-12)


# --- ImageTexture (texture.rs:98-117): a 2x2 binary PPM written by the test -------------------------------
TEXELS = [[(255, 0, 0), (0, 255, 0)], [(0, 0, 255), (51, 102, 204)]]   # [y][x]


def _image_scene(tmp_path):
    path = os.path.join(tmp_path, "kat2x2.ppm")
    with open(path, "wb") as f:
        f.write(b"P6\n2 2\n255\n" + bytes(c for row in TEXELS for px in row for c in px))
    mat = {"type": "Metal", "fuzz": 0.0, "albedo": {"type": "ImageTexture", "image_filename": path}}
    return make_scene([rect(transform=xf((0, 0, 1)))], {"M": mat})


def _image_cases():
    """u' = clamp(u), v' = 1 - clamp(v); x = (u' W) as u32, y = (v' H) as u32; rgb / 255.
    (u, v) = (0.625, 0.75): x = 1.25 -> 1, v' = 0.25, y = 0.5 -> 0 -> texel [0][1] = (0, 255, 0)
    (u, v) = (0.25, 0.25):  x = 0.5 -> 0,  v' = 0.75, y = 1.5 -> 1 -> texel [1][0] = (0, 0, 255)
    (u, v) = (0.625, 0.25): x = 1, y = 1 -> texel [1][1] = (51, 102, 204) -> (0.2, 0.4, 0.8)"""
    return [((0.25, 0.5), TEXELS[0][1]), ((-0.5, -0.5), TEXELS[1][0]), ((0.25, -0.5), TEXELS[1][1])]


def test_oracle_image_texture_lookup(tmp_path):
    sc = _image_scene(str(tmp_path))
    osc = po.OracleScene(sc.desc())
    for (x, y), texel in _image_cases():
        want = tuple((c * (1.0 / 255.0)) * s for c, s in zip(texel, SKY_Z))
        got = osc.trace_pixel_samples(ray((x, y, -3), (0, 0, 1)), 8, seed=SEED, pixel_index=PIXEL)
        assert np.abs(got - np.array(want)).max() <= 1e-15, (got, want)


@pytest.mark.gpu
def test_cuda_image_texture_lookup(tmp_path):
    sc = _image_scene(str(tmp_path))
    for (x, y), texel in _image_cases():
        want = tuple((c * (1.0 / 255.0)) * s for c, s in zip(texel, SKY_Z))
        got = sc.trace_pixel_samples(ray((x, y, -3), (0, 0, 1)), 8, seed=SEED, pixel_index=PIXEL)
        assert_float_path(got, want, 1e-15)


# ------------------------------------------------------------------------------------------------
# (3) the pixel mean (renderer/mod.rs:151-155): (sum of the samples' colours) / samples_number
# ------------------------------------------------------------------------------------------------
def _mean_rays():
    # three rays of one pixel: mirror head-on (albedo x SKY_Z), sky up (0.5, 0.7, 1), sky down (1, 1, 1)
    return np.concatenate([ray((0, 0, -10), (0, 0, 1)), ray((5, 0, 0), (0, 1, 0)), ray((5, 0, 0), (0, -1, 0))])


_MEAN = tuple((a * s + u + 1.0) / 3.0 for a, s, u in zip(ALBEDO, SKY_Z, (0.5, 0.7, 1.0)))


def test_oracle_pixel_mean():
    sc = make_scene([sphere()], {"M": MIRROR})
    got = po.OracleScene(sc.desc()).trace_pixel_samples(_mean_rays(), 8, seed=SEED, pixel_index=PIXEL)
    assert np.abs(got - np.array(_MEAN)).max() <= 1e-15, (got, _MEAN)


@pytest.mark.gpu
def test_cuda_pixel_mean():
    sc = make_scene([sphere()], {"M": MIRROR})
    got = sc.trace_pixel_samples(_mean_rays(), 8, seed=SEED, pixel_index=PIXEL)
    # the mean rebuilt from the three hand-derived ray colours as the device averages them: each path within one ulp
    from test_gpu_caller_rays import check_groups
    cols = np.array([[a * s for a, s in zip(ALBEDO, SKY_Z)], [0.5, 0.7, 1.0], [1.0, 1.0, 1.0]])
    check_groups(got[None], cols, [0, 3], "source pixel mean")
