"""Shading at its decision edges: texture lookups, material branches and the tonemap, against the oracle at float
precision and, where the answer is exact, against an independent numpy expectation.

Frames almost never land on a decision boundary of texture_value, scatter_or_emit or finalize_hit's (u, v).  Every
case here is a crafted caller ray, one ray per group of trace_pixel_samples_group, compared with check_groups: the GPU
colour must be the oracle's FP64 colour rounded to float, or one of that float's two neighbours.  Two facts give exact
control over the inputs:
  * an axis-aligned ray onto an axis-aligned Rectangle (identity rotation and scale, integer translation) hits
    p.x = o.x and p.y = o.y exactly, and the Rectangle's u = (p.x - x0) / (x1 - x0) is o.x when x0 = 0, x1 = 1;
  * rays are never renormalised, so a Dielectric's cos_theta = dot(-rd, n) on such a Rectangle is exactly the chosen
    direction component at bounce level 0.
A DiffuseLight probed at depth 1 returns float(texture_value(u, v, p)).  Material cases run at depths 2 and 8 and end
in the sky.  Every probe set runs once more on new handles under each alternative shading schedule, bit for bit."""
import math

import numpy as np
import pytest

import rs_pathtracing_b200 as rt
from oracle import pyoracle as po

from test_gpu_caller_rays import check_groups
from test_gpu_frame_edges import check_frame
from test_source_kat import make_scene, random_in_unit_sphere, rect, sphere, cube, solid, xf

pytestmark = pytest.mark.gpu

SEED = (1 << 63) + 12345
UP, DOWN = math.inf, -math.inf
ALBEDO = (0.8, 0.4, 0.2)


def light(tex):
    return {"type": "DiffuseLight", "emit": tex}


def rays_along(origins, d):
    o = np.asarray(origins, dtype=np.float64).reshape(-1, 3)
    return np.concatenate([o, np.tile(np.asarray(d, dtype=np.float64), (len(o), 1))], axis=1)


def probe(sc, rays, depth, what, seed=SEED, pix=None):
    """one ray per group; returns (GPU colours, oracle FP64 colours)"""
    rays = np.ascontiguousarray(rays, dtype=np.float64).reshape(-1, 6)
    n = len(rays)
    offsets = np.arange(n + 1, dtype=np.uint64)
    pix = np.arange(n, dtype=np.uint32) if pix is None else np.asarray(pix, dtype=np.uint32)
    cols = po.OracleScene(sc.desc()).group_sample_colors(rays, offsets, pix, depth, seed)
    got = sc.trace_pixel_samples_group(rays, offsets, pix, depth, seed=seed)
    check_groups(got, cols, offsets, what)
    return got, cols


def draw(pix, event, n=1, seed=SEED):
    return po.philox_stream(seed, pix, 0, event, n)


def sky(d):
    t = 0.5 * (d[1] + 1.0)
    return np.array([(1.0 - t) + t * c for c in (0.5, 0.7, 1.0)])


def unit(v):
    v = np.asarray(v, dtype=np.float64)
    return v / math.sqrt(float(v @ v))


# ---- ImageTexture ------------------------------------------------------------------------------------------------

def _texels(w, h):
    """distinct texels: red runs through 37 i + 11 mod 256 (all 256 values when w * h = 256)"""
    i = np.arange(w * h)
    rgb = np.stack([(37 * i + 11) % 256, (91 * i + 5) % 256, 255 - (37 * i + 11) % 256], axis=1)
    return rgb.reshape(h, w, 3).astype(np.uint8)


def _ppm(tmp, w, h):
    path = str(tmp / f"tex_{w}x{h}.ppm")
    with open(path, "wb") as f:
        f.write(b"P6\n%d %d\n255\n" % (w, h) + _texels(w, h).tobytes())
    return {"type": "ImageTexture", "image_filename": path}


def _edges(n):
    """0, 1, and the doubles just below and above k / n for every k"""
    out = {0.0, 1.0}
    for k in range(n + 1):
        out |= {math.nextafter(k / n, DOWN), math.nextafter(k / n, UP)}
    return sorted(x for x in out if 0.0 <= x <= 1.0)


def texel_expected(u, v, w, h):
    """texture.rs:98-117 with the clamp at u = 1 / v = 0: texel / 255"""
    uu = u if math.isnan(u) else min(max(u, 0.0), 1.0)
    vv = 1.0 - (v if math.isnan(v) else min(max(v, 0.0), 1.0))
    fx, fy = uu * w, vv * h
    x = 0 if (math.isnan(fx) or fx <= 0.0) else min(int(fx), w - 1)
    y = 0 if (math.isnan(fy) or fy <= 0.0) else min(int(fy), h - 1)
    return _texels(w, h)[y, x].astype(np.float64) * (1.0 / 255.0)


IMAGE_SIZES = [(1, 1), (1, 7), (7, 1), (3, 5), (256, 1)]


def image_probes(tmp):
    """(name, scene, rays, depth, expected colours or None)"""
    out = []
    for w, h in IMAGE_SIZES:
        sc = make_scene([rect(0.0, 0.0, 1.0, 1.0)], {"M": light(_ppm(tmp, w, h))})
        us, vs = _edges(w), (_edges(h) if w < 256 else [0.0, 0.5, 1.0])
        uv = np.array([(u, v) for u in us for v in vs])
        rays = rays_along(np.c_[uv, np.full(len(uv), -1.0)], (0.0, 0.0, 1.0))
        want = np.array([texel_expected(u, v, w, h) for u, v in uv])
        out.append((f"image {w}x{h} texel edges", sc, rays, 1, want))
    # Cube faces: uv in [-1, 1] (x face: u = p.y, v = p.z), so the clamp at 0 is reached from below.  (A ray along
    # the face at y = +-1 exactly misses: its slab test divides 0 by 0.)
    sc = make_scene([cube()], {"M": light(_ppm(tmp, 3, 5))})
    one = math.nextafter(1.0, DOWN)
    yz = [-one, -0.5, -1e-300, 0.0, 1e-300, 0.2, 1.0 / 3.0, 2.0 / 3.0, 0.6, one]
    pts = np.array([(y, z) for y in yz for z in yz])
    rays = rays_along(np.c_[np.full(len(pts), 3.0), pts], (-1.0, 0.0, 0.0))
    out.append(("image on cube faces", sc, rays, 1, np.array([texel_expected(y, z, 3, 5) for y, z in pts])))
    # Sphere: the seam (p.z = 0, p.x < 0; -p.z = -0 gives atan2 = -pi, u = 0) against p.z = +-1e-300 on either side
    # (u -> 0 or -> 1: columns 0 and 6 of a 7-wide image), and the poles (v = 0, 1; u = 0.5 or 0 by the sign of p.x)
    sc = make_scene([sphere()], {"M": light(_ppm(tmp, 7, 5))})
    seam = [(-3.0, y, z) for y in (0.1, -0.45) for z in (0.0, 1e-300, -1e-300)]
    rays = np.concatenate([rays_along(seam, (1.0, 0.0, 0.0)),
                           rays_along([(0.0, 3.0, 0.0), (-1e-300, 3.0, 0.0), (1e-300, 3.0, 0.0)], (0.0, -1.0, 0.0)),
                           rays_along([(0.0, -3.0, 0.0), (-1e-300, -3.0, 0.0)], (0.0, 1.0, 0.0))])
    out.append(("image on sphere seam and poles", sc, rays, 1, None))
    return out


def test_image_texture_edges(tmp_path):
    for name, sc, rays, depth, want in image_probes(tmp_path):
        got, cols = probe(sc, rays, depth, name)
        if want is not None:
            assert np.array_equal(cols, want), name
    # the seam and the poles: which column and which row, from the oracle's own (u, v)
    name, sc, rays, depth, _ = image_probes(tmp_path)[-1]
    hit = po.OracleScene(sc.desc()).intersect_batch(rays)
    u, v = hit["uv"][:, 0], hit["uv"][:, 1]
    assert (u[[0, 1, 3, 4]] == 0.0).all() and u[1] == 0.0 and (u[[2, 5]] > 0.99).all(), u
    assert list(v[6:9]) == [1.0] * 3 and list(v[9:]) == [0.0] * 2 and list(u[6:]) == [0.5, 0.0, 0.5, 0.5, 0.0], (u, v)
    got, cols = probe(sc, rays, depth, name)
    want = np.array([texel_expected(a, b, 7, 5) for a, b in zip(u, v)])
    assert np.array_equal(cols, want)
    tx = _texels(7, 5)
    assert not np.array_equal(tx[:, 0], tx[:, 6])


# ---- Checker and UVChecker ---------------------------------------------------------------------------------------

ODD, EVEN = (0.1, 0.2, 0.8), (0.9, 0.3, 0.1)
TINY = 5e-324


def checker_probes():
    """Only cases whose sign of the product does not depend on the last bit of any sin: a factor that is exactly
    +-0, or the denormal sin(+-5e-324) = +-5e-324 times factors far from the rounding threshold of the product.
    CheckerTexture, multipliers (1, 1, 1) on the plane z = 1: sines = sin(x) sin(y) sin(1), sin(1) = 0.84.
      x = 0:            +0 * sin(y) -> +0 (y > 0) or -0 (y < 0): not < 0 -> even
      x = +-5e-324:     5e-324 * sin(0.5) = 0.48 denormal ulps -> +-0 -> even;
                        5e-324 * sin(1.5) * sin(1) = 0.84 ulps -> +-5e-324 -> even for +, odd for -
    UVChecker on the unit square, multipliers (2, 1): sines = sin(2 pi v) sin(pi u)
      u = 0:            sin(1.5 pi) * +0 = -0 (v = 0.75) or +0 (v = 0.25) -> even
      u = 5e-324:       sin(pi u) = 1.5e-323 > 0: odd at v = 0.75, even at v = 0.25"""
    tex = {"odd": solid(ODD), "even": solid(EVEN)}
    sc = make_scene([rect(-4.0, -4.0, 4.0, 4.0, transform=xf((0, 0, 1)))],
                    {"M": light(dict(tex, type="CheckerTexture", multipliers=[1, 1, 1]))})
    cases = [((0.0, 0.5), EVEN), ((0.0, -0.5), EVEN), ((-0.0, -0.5), EVEN),
             ((TINY, 0.5), EVEN), ((TINY, -0.5), EVEN), ((-TINY, 0.5), EVEN), ((-TINY, -0.5), EVEN),
             ((TINY, 1.5), EVEN), ((-TINY, 1.5), ODD), ((TINY, -1.5), ODD), ((-TINY, -1.5), EVEN),
             ((0.5, 0.0), EVEN), ((-0.5, 0.0), EVEN), ((-0.5, 0.5), ODD)]
    xy = np.array([c[0] for c in cases])
    out = [("checker signed zeros", sc, rays_along(np.c_[xy, np.full(len(xy), -1.0)], (0.0, 0.0, 1.0)), 1,
            np.array([c[1] for c in cases]))]
    sc = make_scene([rect(0.0, 0.0, 1.0, 1.0)], {"M": light(dict(tex, type="UVChecker", multipliers=[2, 1]))})
    cases = [((0.0, 0.75), EVEN), ((0.0, 0.25), EVEN), ((TINY, 0.75), ODD), ((TINY, 0.25), EVEN),
             ((0.5, 0.0), EVEN), ((0.5, 0.75), ODD)]
    uv = np.array([c[0] for c in cases])
    out.append(("uv checker signed zeros", sc, rays_along(np.c_[uv, np.full(len(uv), -1.0)], (0.0, 0.0, 1.0)), 1,
                np.array([c[1] for c in cases])))
    # exactly RT_TEX_MAX_DEPTH = 8 nested levels, alternating kinds: the leaf's colour, not black
    leaf = solid((0.2, 0.4, 0.8))
    t = leaf
    for k in range(8):
        t = ({"type": "CheckerTexture", "multipliers": [1, 1, 1]} if k % 2 else
             {"type": "UVChecker", "multipliers": [1, 1]}) | {"odd": t, "even": t}
    sc = make_scene([rect(0.0, 0.0, 1.0, 1.0)], {"M": light(t)})
    uv = np.array([(0.3, 0.6), (0.0, 0.0), (0.9, 0.1)])
    out.append(("8 nested checkers", sc, rays_along(np.c_[uv, np.full(3, -1.0)], (0.0, 0.0, 1.0)), 1,
                np.tile([0.2, 0.4, 0.8], (3, 1))))
    return out


def test_checker_edges():
    for name, sc, rays, depth, want in checker_probes():
        got, cols = probe(sc, rays, depth, name)
        assert np.array_equal(cols, want), name


# ---- NoiseTexture ------------------------------------------------------------------------------------------------

I31 = 2.0 ** 31
NOISE_COORDS = [0.0, 1.0, -1.0, 7.0, math.nextafter(1.0, DOWN), math.nextafter(1.0, UP), math.nextafter(7.0, DOWN),
                math.nextafter(-1.0, UP), math.nextafter(-1.0, DOWN), -0.5, -3.25, 255.0, 256.0, 255.0 / 256.0,
                math.nextafter(256.0, DOWN), -1.0 / 256.0, I31 - 2, I31 - 1, -(I31 - 1), I31, -I31, I31 + 1,
                -(I31 + 1), -(I31 + 2), 1e12, -1e12, 1e300, -1e300]
NOISE_PLANES = [0.0, -1.0, 255.0, 256.0, I31 - 1, -I31, 1e12]


def noise_reference(pn, p):
    """Perlin::noise (src/algebra/noise.rs:43-73) transcribed on Python floats: floor, `as i32` (saturating), the
    & 255 wrap, the Hermite weights and the eight corner terms summed in multi_cartesian_product order"""
    def as_i32(v):
        return 0 if v != v else int(max(min(v, 2147483647.0), -2147483648.0))
    f = [math.floor(c) for c in p]
    i = [as_i32(float(c)) for c in f]
    uvw = [c - float(fc) for c, fc in zip(p, f)]
    h = [t * t * (3.0 - 2.0 * t) for t in uvw]
    perms = (pn.perm_x, pn.perm_y, pn.perm_z)
    acc = 0.0
    for a in range(2):
        for b in range(2):
            for c in range(2):
                d = (a, b, c)
                g = pn.ranvec[perms[0][(i[0] + a) & 255] ^ perms[1][(i[1] + b) & 255] ^ perms[2][(i[2] + c) & 255]]
                dot = g.x * (uvw[0] - a) + g.y * (uvw[1] - b) + g.z * (uvw[2] - c)
                w = 1.0
                for k in range(3):
                    w = w * ((float(d[k]) * h[k] + float(1 - d[k]) * (1.0 - h[k])))
                acc = acc + w * dot
    return acc


def noise_probes():
    out = []
    tex = {"type": "NoiseTexture", "scale": 3.0}
    cs = NOISE_COORDS
    xy = [(c, 0.37) for c in cs] + [(-2.6, c) for c in cs] + [(c, c) for c in cs[::3]]
    for z in NOISE_PLANES:
        sc = make_scene([rect(-1e301, -1e301, 1e301, 1e301, transform=xf((0, 0, z)))], {"M": light(tex)})
        rays = rays_along([(x, y, z - 1.0) for x, y in xy], (0.0, 0.0, 1.0))
        out.append((f"noise on z = {z}", sc, rays, 1, None))
    return out


def test_noise_edges():
    for name, sc, rays, depth, _ in noise_probes():
        osc = po.OracleScene(sc.desc())
        hit = osc.intersect_batch(rays)
        want_p = rays[:, :3].copy()
        want_p[:, 2] += 1.0
        assert np.array_equal(hit["point"], want_p), name    # the probe lands exactly on p
        pn = sc.desc().noise[0]
        for p in want_p:
            assert po.perlin_noise(pn, p) == noise_reference(pn, [float(c) for c in p]), (name, p)
        probe(sc, rays, depth, name)


def test_noise_reference_in_all_three_coordinates():
    """the oracle's saturation and wrap, checked in z as well (the probes above hold z to a few planes)"""
    sc = noise_probes()[0][1]
    pn = sc.desc().noise[0]
    rng = np.random.default_rng(3)
    for k in range(400):
        p = [float(rng.choice(NOISE_COORDS)) for _ in range(3)]
        assert po.perlin_noise(pn, p) == noise_reference(pn, p), p


# ---- Dielectric --------------------------------------------------------------------------------------------------

def reflectance(c, ratio):
    r0 = (1.0 - ratio) / (1.0 + ratio)
    r0 = r0 * r0
    x = 1.0 - c
    x2 = x * x
    return r0 + (1.0 - r0) * (x * (x2 * x2))


def _glass(ior):
    return make_scene([rect(-1e7, -1e7, 1e7, 1e7)], {"M": {"type": "Dielectric", "index_of_refraction": ior}})


def _slanted(c, front):
    """a ray in the y-z plane through (0, 0, 0) with direction (0, s, -+c), s = sqrt(1 - c^2) (or 1 when c > 1): on the
    plane z = 0, cos_theta = c exactly, front face when coming down from z > 0"""
    s = math.sqrt(max(1.0 - c * c, 0.0)) if c <= 1.0 else 0.0
    dz = -c if front else c
    return np.array([0.0, -s, -dz, 0.0, s, dz])


def _pixels_with_draw(lo, hi, n, event=1, start=0):
    out, p = [], start
    while len(out) < n:
        if lo < draw(p, event)[0] < hi:
            out.append(p)
        p += 1
    return out


def dielectric_probes():
    out = []
    # total internal reflection on the back face (ratio = ior): ratio * sqrt(1 - c c) around 1
    tir = [(2.0, 0.8660254037844386, 1.0000000000000002), (2.0, 0.8660254037844387, 0.9999999999999998),
           (1.25, 0.5999999999999998, 1.0000000000000004), (1.25, 0.5999999999999999, 1.0), (1.25, 0.6, 1.0),
           (1.25, 0.6000000000000001, 0.9999999999999999)]
    pix = _pixels_with_draw(0.5, 1.0, 1)
    for ior, c, prod in tir:
        assert ior * math.sqrt(1.0 - c * c) == prod
        out.append((f"TIR ior {ior} cos {c!r}", _glass(ior), _slanted(c, False)[None], 8, None, pix, prod > 1.0))
    # the Fresnel draw: adjacent cos doubles around reflectance(cos, 1/1.5) == draw, front face, draw of event 1
    ratio = 1.0 / 1.5
    rays, pix, refl = [], [], []
    for p in _pixels_with_draw(0.06, 0.9, 96, start=1000):
        u = draw(p, 1)[0]
        lo, hi = 0.0, 1.0                      # reflectance(lo) > u >= reflectance(hi); bisect down to adjacent doubles
        while math.nextafter(lo, UP) < hi:
            mid = 0.5 * (lo + hi)
            if mid in (lo, hi):
                mid = math.nextafter(lo, UP)
            lo, hi = (mid, hi) if reflectance(mid, ratio) > u else (lo, mid)
        for c in (lo, hi):
            rays.append(_slanted(c, True))
            pix.append(p)
            refl.append(reflectance(c, ratio) > u)
    assert any(refl) and not all(refl)
    out.append(("Fresnel draw edges", _glass(1.5), np.array(rays), 2, None, pix, refl))
    # cos exactly 1, just above 1 (sqrt of a negative: NaN), tiny; ior 1, below 1, huge and 0 (a NaN path)
    cs = [1.0, math.nextafter(1.0, UP), 0.6, 1e-6]
    for ior in (1.5, 1.0, 0.5, 1e300, 0.0):
        rays = np.array([_slanted(c, f) for c in cs for f in (True, False)])
        out.append((f"glass ior {ior}", _glass(ior), rays, 8, None, list(range(len(rays))), None))
    return out


def test_dielectric_edges():
    for name, sc, rays, depth, _, pix, refl in dielectric_probes():
        got, cols = probe(sc, rays, depth, name, pix=pix)
        if refl is None:
            continue
        # reflected: direction (0, s, +-c) -> the sky at y = s; refracted at these angles: y = ratio s / |...|
        for r, c, want_reflect in zip(rays, cols, np.broadcast_to(refl, len(rays))):
            assert np.allclose(c, sky(unit(r[3:] * (1, 1, -1))), rtol=0, atol=1e-14) == bool(want_reflect), (name, r)


# ---- Lambertian --------------------------------------------------------------------------------------------------

def lambertian_probes():
    """a ray aimed at the unit-sphere point -u, where u is the path's random_unit draw at bounce level 0 (event 1):
    the normal there is -u up to rounding, normal + u is below approx_zero's 1e-15 in every component, and the
    scattered direction must fall back to the normal"""
    rays, pix = [], []
    for p in range(64):
        u = np.array(unit(random_in_unit_sphere(draw(p, 1, 96))))
        rays.append(np.r_[-3.0 * u, u])
        pix.append(p)
    sc = make_scene([sphere()], {"M": {"type": "Lambertian", "albedo": solid(ALBEDO)}})
    return [("Lambertian fallback", sc, np.array(rays), 8, None, pix)]


def test_lambertian_fallback():
    name, sc, rays, depth, _, pix = lambertian_probes()[0]
    hit = po.OracleScene(sc.desc()).intersect_batch(rays)
    n = hit["normal"]
    u = rays[:, 3:]
    small = (np.abs(n + u) < 1e-15).all(axis=1)
    assert small.sum() >= 16, small.sum()
    got, cols = probe(sc, rays[small], depth, name, pix=np.array(pix)[small])
    for c, nn in zip(cols, n[small]):
        assert np.allclose(c, np.array(ALBEDO) * sky(unit(nn)), rtol=0, atol=1e-15), (c, nn)


# ---- Metal -------------------------------------------------------------------------------------------------------

def metal_probes():
    out = []
    d = unit([0.3, -0.2, 1.0])
    rays = np.concatenate([rays_along([(0.0, 0.0, -5.0), (0.0, 0.5, -5.0), (0.5, 0.0, -5.0)], (0.0, 0.0, 1.0)),
                           rays_along([(5.0, -0.0, 0.0), (-0.0, -5.0, 0.0)], (-1.0, 0.0, -0.0)),
                           rays_along([(0.0, -5.0, 0.0)], (-0.0, 1.0, 0.0)),
                           np.r_[-5.0 * d, d][None]])
    for fuzz in (0.0, -0.0, 1e-300, -0.5, 0.5, 3.0):
        sc = make_scene([sphere()], {"M": {"type": "Metal", "albedo": solid(ALBEDO), "fuzz": fuzz}})
        out.append((f"metal fuzz {fuzz!r}", sc, rays, 8, None, None))
    # fuzz 3 with a unit-ball draw that points into the sphere: the scattered ray starts into the surface
    pix = [p for p in range(200) if -(np.array(random_in_unit_sphere(draw(p, 1, 96)))[2]) * 3.0 < -1.2][:8]
    assert len(pix) >= 4
    sc = make_scene([sphere()], {"M": {"type": "Metal", "albedo": solid(ALBEDO), "fuzz": 3.0}})
    out.append(("metal fuzz 3 into the surface", sc, rays_along([(0.0, 0.0, -5.0)] * len(pix), (0.0, 0.0, 1.0)), 8,
                None, pix))
    # a mirror cube hit exactly on edges and corners: the normal (tie order x, y, z) decides the reflection
    sc = make_scene([cube()], {"M": {"type": "Metal", "albedo": solid(ALBEDO), "fuzz": 0.0}})
    out.append(("mirror cube edges", sc, CUBE_RAYS, 8, None, None))
    return out


def test_metal_edges():
    mirror = None
    for name, sc, rays, depth, _, pix in metal_probes():
        got, cols = probe(sc, rays, depth, name, pix=pix)
        if name in ("metal fuzz 0.0", "metal fuzz -0.0", "metal fuzz 1e-300"):
            # -0.0 takes the mirror branch; 1e-300 * ball vanishes against the reflected direction
            mirror = got if mirror is None else mirror
            assert np.array_equal(got, mirror), name
        if name == "metal fuzz -0.5":
            assert not np.array_equal(got, mirror), "negative fuzz is not a mirror"


# ---- Cube normals ------------------------------------------------------------------------------------------------

CUBE_RAYS = np.array([
    [3, 3, 0.3, -1, -1, 0], [3, -3, 0.3, -1, 1, 0], [-3, 3, -0.3, 1, -1, 0], [-3, -3, 0.3, 1, 1, 0],
    [0.3, 3, 3, 0, -1, -1], [3, 0.3, 3, -1, 0, -1], [3, 0.3, -3, -1, 0, 1],
    [3, 3, 3, -1, -1, -1], [-3, 3, -3, 1, -1, 1], [3, -3, -3, -1, 1, 1],
    [0, 0, 0.3, 1, 1, 0], [0, 0, 0, 1, 1, 1], [0, 0, 0, -1, 1, -1], [0.3, 0, 0, 0, -1, -1],
    [3, 0, 0, -1, 0, 0], [3, -0.0, -0.0, -1, 0, 0], [-0.0, 3, 0, 0, -1, 0], [0, 0, -3, -0.0, -0.0, 1],
], dtype=np.float64)


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


@pytest.mark.parametrize("mode", [rt._ffi.RT_ISECT_BRUTE, rt._ffi.RT_ISECT_FAST])
def test_cube_edge_and_corner_normals(mode):
    """normal, point and front face by bit pattern (so +0 and -0 differ), uv exactly; and the face the tie order
    max_c == ax, then ay, then az picks"""
    sc = make_scene([cube()])
    want = po.OracleScene(sc.desc()).intersect_batch(CUBE_RAYS)
    got = sc.closest_hit(CUBE_RAYS, mode=mode)
    assert np.array_equal(got["index"], want["index"]) and (want["index"] == 0).all()
    for k in ("t", "normal", "point", "uv"):
        assert np.array_equal(_bits(got[k]), _bits(want[k])), (k, got[k], want[k])
    assert np.array_equal(got["front"], want["front"])
    p = want["point"]
    a = np.abs(p)
    face = np.where(a[:, 0] == a.max(axis=1), 0, np.where(a[:, 1] == a.max(axis=1), 1, 2))
    n_obj = np.zeros((len(p), 3))
    n_obj[np.arange(len(p)), face] = np.sign(p[np.arange(len(p)), face])
    flip = np.where(want["front"] == 1, 1.0, -1.0)[:, None]
    assert np.array_equal(want["normal"], n_obj * flip), (want["normal"], n_obj * flip)
    assert face[0] == 0 and face[4] == 1 and face[7] == 0


# ---- every probe set under every shading schedule, and one frame --------------------------------------------------

def _all_probes(tmp):
    out = []
    for name, sc, rays, depth, *rest in image_probes(tmp) + checker_probes() + noise_probes():
        out.append((name, sc, rays, depth, None))
    for name, sc, rays, depth, _, pix, *rest in dielectric_probes() + lambertian_probes() + metal_probes():
        out.append((name, sc, rays, depth, pix))
    return out


SCHEDULES = [{"RT_B200_FUSED_BOUNCE": "1"}, {"RT_B200_SHADE_BINNED": "0"}, {"RT_B200_SHADE_BINNED": "1"}]


def test_schedules_give_the_same_colours(tmp_path, monkeypatch):
    base = []
    for name, sc, rays, depth, pix in _all_probes(tmp_path):
        base.append(probe(sc, rays, depth, name, pix=pix)[0])
    for env in SCHEDULES:
        with monkeypatch.context() as m:
            for k, v in env.items():
                m.setenv(k, v)
            for (name, sc, rays, depth, pix), ref in zip(_all_probes(tmp_path), base):   # new handles read the variables
                n = len(rays)
                pix = np.arange(n, dtype=np.uint32) if pix is None else np.asarray(pix, dtype=np.uint32)
                got = sc.trace_pixel_samples_group(rays, np.arange(n + 1, dtype=np.uint64), pix, depth, seed=SEED)
                assert np.array_equal(got, ref, equal_nan=True), (env, name)


def test_edge_material_frame(tmp_path):
    """one 48x32 frame of a scene built from these materials, no pixel exempt"""
    shapes = [cube(xf((-2.2, -0.6, 1.0), (0.8, 0.8, 0.8), (0, 30, 0)), "MIRROR"),
              sphere(xf((0.0, 0.2, 0.0), (1.1, 1.1, 1.1)), "GLASS"),
              rect(-10.0, -10.0, 10.0, 10.0, xf((0, -1.2, 0), (1, 1, 1), (90, 0, 0)), "NOISE"),
              rect(0.0, 0.0, 1.0, 1.0, xf((1.4, -0.5, 0.5), (1.5, 1.5, 1.5)), "IMAGE"),
              sphere(xf((2.3, 0.8, 1.5), (0.7, 0.7, 0.7)), "CHECK"),
              sphere(xf((0.0, 4.0, 2.0), (1.0, 1.0, 1.0)), "LIGHT")]
    mats = {"MIRROR": {"type": "Metal", "albedo": solid(ALBEDO), "fuzz": -0.0},
            "GLASS": {"type": "Dielectric", "index_of_refraction": 2.0},
            "NOISE": {"type": "Lambertian", "albedo": {"type": "NoiseTexture", "scale": 4.0}},
            "IMAGE": {"type": "Metal", "albedo": _ppm(tmp_path, 3, 5), "fuzz": 3.0},
            "CHECK": {"type": "Lambertian", "albedo": {"type": "UVChecker", "multipliers": [4, 8],
                                                       "odd": solid(ODD), "even": solid(EVEN)}},
            "LIGHT": light(solid((4.0, 4.0, 4.0)))}
    sc = make_scene(shapes, mats)
    cam = sc.camera()
    w, h, spp, depth, seed = 48, 32, 2, 8, SEED
    frame = rt.GpuRenderer(sc, 1, depth, seed=seed).render(cam, w, h, spp)
    check_frame(frame, po.OracleScene(sc.desc()), cam, w, h, spp, depth, seed, "edge materials frame")


# ---- tonemap -----------------------------------------------------------------------------------------------------

def test_tonemap_edges():
    """k_tonemap against sqrt, clamp(0, 0.999), * 256, `as u8` (NaN -> 0) at the truncation edges: x = (k/256)^2 and its
    float neighbours for every k, 0.999^2 and its neighbours, signed zeros, negatives, infinities, NaN, subnormals"""
    xs = []
    for k in range(257):
        x = (k / 256.0) ** 2
        xs += [math.nextafter(x, DOWN), x, math.nextafter(x, UP)]
    x = 0.999 * 0.999
    xs += [math.nextafter(math.nextafter(x, DOWN), DOWN), math.nextafter(x, DOWN), x, math.nextafter(x, UP)]
    xs += [0.0, -0.0, -1e-300, -1.0, -math.inf, math.inf, math.nan, 5e-324, 2.2250738585072014e-308, 1e300]
    v = np.array(xs)
    frame = np.stack([v, np.roll(v, 1), np.roll(v, 2)], axis=1).reshape(-1, 1, 3)
    sc = make_scene([sphere()])
    got = rt.tonemap_rgba8(sc, frame).reshape(-1, 4)
    with np.errstate(invalid="ignore"):
        q = np.clip(np.sqrt(frame.reshape(-1, 3)), 0.0, 0.999) * 256.0
    want = np.where(np.isnan(q), 0.0, q).astype(np.uint8)
    assert np.array_equal(got[:, :3], want) and (got[:, 3] == 255).all()
    assert {0, 1, 127, 128, 254, 255} <= set(want[:, 0].tolist())
