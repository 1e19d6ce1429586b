"""Random scenes over the whole scene-JSON schema (every shape kind incl. the six ray-marched surfaces with
anisotropic / rotated transforms, inverse_normal spheres, every material, nested textures incl. Perlin
noise): nearest hit bit-exact against the oracle (both kernels), RT_ISECT_VERIFY clean, and a small frame
path for path.  Seeds are fixed; a failure prints the seed."""
import json

import numpy as np
import pytest

import rs_pathtracing_b200 as rt
from oracle import pyoracle as po

from test_gpu_frame_edges import check_frame
from test_gpu_intersect import SURFACES, _compare

pytestmark = pytest.mark.gpu


def random_scene(seed):
    rng = np.random.default_rng(seed)
    u = lambda a, b: float(rng.uniform(a, b))
    col = lambda: [u(0.05, 1.0), u(0.05, 1.0), u(0.05, 1.0)]

    def texture(depth=0):
        kinds = ["SolidColor", "SolidColor", "CheckerTexture", "UVChecker", "NoiseTexture"]
        k = kinds[rng.integers(0, len(kinds) if depth < 2 else 2)]
        if k == "SolidColor":
            return {"type": k, "color": col()}
        if k == "CheckerTexture":
            return {"type": k, "odd": texture(depth + 1), "even": texture(depth + 1), "multipliers": [u(0.5, 4), u(0.5, 4), u(0.5, 4)]}
        if k == "UVChecker":
            return {"type": k, "odd": texture(depth + 1), "even": texture(depth + 1), "multipliers": [u(1, 12), u(1, 12)]}
        return {"type": k, "scale": u(0.5, 6)}

    materials = {}
    for i in range(8):
        k = ["Lambertian", "Lambertian", "Metal", "Metal", "Dielectric", "DiffuseLight", "Lambertian", "EmptyMaterial"][i]
        if k == "Lambertian":
            materials[f"m{i}"] = {"type": k, "albedo": texture()}
        elif k == "Metal":
            materials[f"m{i}"] = {"type": k, "albedo": texture(), "fuzz": [0.0, u(0.05, 1.0)][i % 2]}
        elif k == "Dielectric":
            materials[f"m{i}"] = {"type": k, "index_of_refraction": u(1.1, 2.2)}
        elif k == "DiffuseLight":
            materials[f"m{i}"] = {"type": k, "emit": {"type": "SolidColor", "color": [u(1, 8)] * 3}}
        else:
            materials[f"m{i}"] = {"type": k}
    tr = lambda c, s: {"translate": [float(x) for x in c], "rotate": [u(-180, 180), u(-180, 180), u(-180, 180)],
                       "scale": [float(x) for x in s]}
    shapes = []
    for i in range(int(rng.integers(6, 30))):
        c = rng.uniform(-6, 6, 3)
        m = f"m{rng.integers(0, 8)}"
        kind = rng.integers(0, 4)
        if kind == 0:
            s = rng.uniform(0.3, 1.5) * np.array([1.0, u(0.5, 2.0), u(0.5, 2.0)])
            shapes.append({"type": "Sphere", "name": f"s{i}", "material": m, "transform": tr(c, s),
                           "inverse_normal": bool(rng.integers(0, 5) == 0)})
        elif kind == 1:
            shapes.append({"type": "Cube", "name": f"c{i}", "material": m, "transform": tr(c, rng.uniform(0.2, 1.2, 3))})
        elif kind == 2:
            x0, y0 = u(-3, 0), u(-3, 0)
            shapes.append({"type": "Rectangle", "x0": x0, "y0": y0, "x1": x0 + u(0.5, 5), "y1": y0 + u(0.5, 5),
                           "material": m, "transform": tr(c, rng.uniform(0.5, 2.0, 3))})
        else:
            surf = list(SURFACES)[rng.integers(0, len(SURFACES))]
            sc = u(0.4, 1.5)
            shapes.append({"type": "BruteForsableShape", "shape": SURFACES[surf], "step": [0.01, 0.02, 0.004][rng.integers(0, 3)],
                           "depth": int(rng.integers(2, 5)), "material": m,
                           "transform": tr(c, [sc, sc * u(0.7, 1.4), sc * u(0.7, 1.4)])})
    shapes.append({"type": "Sphere", "name": "ground", "material": "m0",
                   "transform": {"translate": [0, -1008, 0], "rotate": [0, 0, 0], "scale": [1000, 1000, 1000]}})
    pos = rng.uniform(-1, 1, 3)
    pos = pos / np.linalg.norm(pos) * u(14, 22)
    pos[1] = abs(pos[1])
    return {"camera": {"position": pos.tolist(), "direction": (-pos).tolist(), "up": [0, 1, 0], "fov": 40.0, "focal_length": 1.0},
            "background": [0, 0, 0], "materials": materials, "shapes": shapes}


def rays_for(sc, cam, n, rng):
    prim = np.array([po.get_ray(cam, 64, 64, x, y) for x, y in zip(rng.uniform(0, 64, n // 2), rng.uniform(0, 64, n // 2))])
    a = rng.uniform(-8, 8, (n - n // 2, 3))
    b = rng.uniform(-6, 6, (n - n // 2, 3))
    return np.concatenate([prim, rt.make_rays(a, b - a)])


@pytest.mark.parametrize("seed", range(12))
def test_random_scene_parity(seed):
    data = json.dumps(random_scene(1000 + seed))
    sc = rt.Scene.from_json(data, add_random_spheres=(seed % 3 == 0), random_spheres_seed=seed + 1)
    cam = sc.camera()
    osc = po.OracleScene(sc.desc())
    rng = np.random.default_rng(seed)
    rays = rays_for(sc, cam, 3000, rng)
    want = osc.intersect_batch(rays)
    assert (want["index"] >= 0).mean() > 0.3, f"seed {seed}: degenerate scene"
    for mode in (rt.RT_ISECT_BRUTE, rt.RT_ISECT_FAST):
        _compare(sc.closest_hit(rays, mode=mode), want, len(rays), mode)
    sc.reset_stats()
    sc.closest_hit(rays, mode=rt.RT_ISECT_VERIFY, want=("index",))
    st = sc.stats()
    assert st.verify_rays == 0 and st.verify_false_culls == 0, f"seed {seed}"
    w, h, spp, depth = 40, 30, 3, 6
    got = rt.GpuRenderer(sc, 12, depth, seed=seed).render(cam, w, h, spp)
    check_frame(got, osc, cam, w, h, spp, depth, seed, f"random scene {seed}")   # no pixel exempt
