"""Occlusion queries (rt_occluded_batch[_device]) bit for bit against the nearest hit.

occluded[i] must be exactly `rt_intersect_batch(RT_ISECT_BRUTE)(ray i, t_min, tmax_i).index != -1` in every mode: the
literal loop's max_t only shrinks at an acceptance, so it reports a hit iff some shape accepts the ray at tmax_i, and
the any-hit query may stop at the first shape that does.  The reference here is always the nearest hit of the device's
literal loop with each ray's own bound; on every non-Torus scene a subset is also checked against the oracle."""
import ctypes as C
import json
import math

import numpy as np
import pytest

import rs_pathtracing_b200 as rt
from rs_pathtracing_b200 import _ffi, api
from oracle import pyoracle as po

from conftest import scene_path
from test_cull_cpu import big_scene, box_rays
from test_gpu_frame_edges import marched_scene
from test_gpu_intersect import TRIO, bench_rays
from test_gpu_render import _variant_4b
from test_gpu_scene_update import Edited, create, update_transforms

pytestmark = pytest.mark.gpu

MODES = (rt.RT_ISECT_BRUTE, rt.RT_ISECT_FAST, rt.RT_ISECT_VERIFY)

DEGENERATE = {   # test_gpu_intersect.py's degenerate-ray scene: D == 0 tangents, a Cube around the origin, NaN t
    "shapes": [
        {"type": "Rectangle", "x0": -1, "y0": -1, "x1": 1, "y1": 1, "material": "M",
         "transform": {"translate": [0, 0, 5], "rotate": [0, 0, 0], "scale": [1, 1, 1]}},
        {"type": "Cube", "name": "c", "material": "M",
         "transform": {"translate": [10, 0, 0], "rotate": [0, 0, 0], "scale": [1, 1, 1]}},
        {"type": "Sphere", "name": "s", "material": "M",
         "transform": {"translate": [0, 0, 0], "rotate": [0, 0, 0], "scale": [1, 1, 1]}},
        {"type": "Sphere", "name": "s2", "material": "M",
         "transform": {"translate": [0, 0, 20], "rotate": [0, 0, 0], "scale": [2, 2, 2]}},
    ]}
DEGENERATE_RAYS = np.array([
    [1.0, 0.0, -10.0, 0.0, 0.0, 1.0],      # tangent to the unit sphere: D == 0
    [2.0, 0.0, -10.0, 0.0, 0.0, 1.0],      # tangent to the scaled sphere behind it
    [-10.0, 1.0, 0.0, -1.0, 0.0, 0.0],     # tangent to the unit sphere pointing away: D == 0 accepted at t = -10
    [10.0, 0.2, 0.1, 0.0, 0.0, 1.0],       # origin inside the cube
    [-5.0, 0.0, 5.0, 1.0, 0.0, 0.0],       # in the rectangle's plane: t = -0/0 = NaN
    [0.0, 0.0, -10.0, 0.0, 0.0, 1.0],      # plain hit through everything
])

SCENES = ["trio", "degenerate", "spheres.json", "cornell_box.json", "dupin.json", "cube_test.json", "light_source.json",
          "detached_materials.json", "torus.json", "4b", "march33", "big"]

_cache = {}


def load(name):
    """(scene, camera, has a Torus)"""
    if name not in _cache:
        if name in ("trio", "degenerate"):
            scene = json.loads(json.dumps(TRIO))
            if name == "degenerate":
                scene["shapes"] = DEGENERATE["shapes"]
            sc = rt.Scene.from_json(json.dumps(scene), add_random_spheres=False)
            cam = sc.camera()
        elif name == "march33":
            sc = rt.Scene.from_json(json.dumps(marched_scene(33)), add_random_spheres=False)
            cam = sc.camera()
        elif name == "big":
            sc = big_scene(10000, seed=5, extent=25.0)
            cam = rt.camera_new((0, 0, -80), (0, 0, 1), (0, 1, 0), 1.0, 0.8)
        elif name == "4b":
            sc = rt.Scene.from_file(scene_path("detached_materials.json"), random_spheres_seed=1)
            cam = _variant_4b(sc)
        else:
            sc = rt.Scene.from_file(scene_path(name), random_spheres_seed=1)
            cam = sc.camera()
        _cache[name] = (sc, cam)
    sc, cam = _cache[name]
    return sc, cam, bool((sc.shape_kinds() == _ffi.RT_SHAPE_TORUS).any())


def nearest(sc, rays, t_min, t_max):
    return sc.closest_hit(rays, t_min, t_max, mode=rt.RT_ISECT_BRUTE, want=("index", "t", "point", "normal"))


def reference(sc, rays, t_min, t_max):
    """BRUTE's index != -1 with each ray's own bound (rays grouped by the bits of their bound)"""
    if np.isscalar(t_max):
        return nearest(sc, rays, t_min, t_max)["index"] >= 0
    out = np.empty(len(rays), bool)
    keys = np.ascontiguousarray(t_max).view(np.uint64)
    for k in np.unique(keys):
        sel = keys == k
        out[sel] = nearest(sc, rays[sel], t_min, float(np.array([k], np.uint64).view(np.float64)[0]))["index"] >= 0
    return out


def assert_occluded(sc, rays, t_min=0.001, t_max=math.inf, want=None, modes=MODES):
    rays = np.ascontiguousarray(rays, np.float64)
    if want is None:
        want = reference(sc, rays, t_min, t_max)
    for mode in modes:
        sc.reset_stats()
        got = sc.occluded(rays, t_min, t_max, mode=mode)
        assert got.dtype == np.bool_ and got.shape == (len(rays),)
        bad = np.flatnonzero(got != want)
        assert bad.size == 0, f"mode {mode}: {bad.size} of {len(rays)} differ, first rays {rays[bad[:3]].tolist()}"
        if mode == rt.RT_ISECT_VERIFY:
            st = sc.stats()
            assert (st.verify_rays, st.verify_false_culls) == (0, 0)
    return want


def unit(v):
    return v / np.linalg.norm(v, axis=1, keepdims=True)


def world_rays(desc, index, o_obj, d_obj):
    """object-space rays of shapes `index` in world space (direct rows of the description)"""
    m = np.ctypeslib.as_array(desc.direct, shape=(desc.n_shapes, 12))[index].reshape(-1, 3, 4)
    o = np.einsum("kij,kj->ki", m[:, :, :3], o_obj) + m[:, :, 3]
    d = np.einsum("kij,kj->ki", m[:, :, :3], d_obj)
    return np.concatenate([o, d], axis=1)


def light_points(sc, rng, n):
    """uniform points of the scene's DiffuseLight shapes' object-space unit squares / spheres, or shape centres"""
    d = sc.desc()
    mats = [d.materials[d.material[i]].kind for i in range(d.n_shapes)]
    lights = [i for i in range(d.n_shapes) if mats[i] == _ffi.RT_MAT_DIFFUSE_LIGHT and d.kind[i] != _ffi.RT_SHAPE_MARCH]
    pool = lights or list(range(min(d.n_shapes, 64)))
    idx = np.array(pool)[rng.integers(0, len(pool), n)]
    obj = np.zeros((n, 3))
    kinds = np.array([d.kind[i] for i in idx])
    params = np.ctypeslib.as_array(d.params, shape=(d.n_shapes, 8))[idx]
    rect = kinds == _ffi.RT_SHAPE_RECTANGLE
    u = rng.uniform(0, 1, (n, 2))
    obj[rect, 0] = params[rect, 0] + u[rect, 0] * (params[rect, 2] - params[rect, 0])
    obj[rect, 1] = params[rect, 1] + u[rect, 1] * (params[rect, 3] - params[rect, 1])
    obj[~rect] = unit(rng.normal(size=((~rect).sum(), 3))) * 0.999
    return world_rays(d, idx, obj, np.zeros((n, 3)))[:, :3]


def ray_sets(sc, cam, seed=0):
    """the ray sets of the issue, as a dict name -> (rays, t_min, t_max)"""
    rng = np.random.default_rng(seed)
    d = sc.desc()
    n_shapes = d.n_shapes
    kinds = sc.shape_kinds()
    out = {"cfg2": (bench_rays(2048, seed=seed), 0.001, math.inf)}
    w, h = 320, 240
    cam_rays = np.array([po.get_ray(cam, w, h, x, y) for x, y in rng.uniform(0, 1, (1024, 2)) * (w, h)])
    out["camera"] = (cam_rays, 0.001, math.inf)
    hits = nearest(sc, cam_rays, 0.001, math.inf)
    hit = hits["index"] >= 0
    pts, nrm = hits["point"][hit], hits["normal"][hit]
    if len(pts):
        dirs = unit(nrm + unit(rng.normal(size=pts.shape)))
        out["secondary"] = (np.concatenate([pts, dirs], 1), 0.001, math.inf)
        lp = light_points(sc, rng, len(pts))
        srays, dist = api.shadow_rays(pts, lp)
        ok = dist > 0
        out["shadow"] = (srays[ok], 0.001, (1 - 1e-9) * dist[ok])
    # from inside shapes: the centre of a few Spheres (Dielectric ones included), Cubes and marched bounding balls
    inside = rng.choice(n_shapes, size=min(n_shapes, 200), replace=False)
    out["inside"] = (world_rays(d, inside, rng.uniform(-0.3, 0.3, (len(inside), 3)),
                                unit(rng.normal(size=(len(inside), 3)))), 0.001, math.inf)
    # axis-aligned directions with signed zeros, from the camera and from shape centres
    axes = []
    for a in range(3):
        for s in (1.0, -1.0):
            for z in (0.0, -0.0):
                v = [z, z, z]
                v[a] = s
                axes.append(v)
    origins = np.concatenate([[cam.position.tuple()], world_rays(d, inside[:8], np.zeros((min(8, len(inside)), 3)),
                                                                 np.zeros((min(8, len(inside)), 3)))[:, :3]])
    out["axes"] = (np.array([list(o) + v for o in origins for v in axes]), 0.001, math.inf)
    # Sphere tangents (object space (1, 0, -10) along +z: D == 0 up to the rounding of the transform) and Rectangle rays
    # in the shape's plane (o.z = d.z = 0 in object space)
    sph = np.flatnonzero(kinds == _ffi.RT_SHAPE_SPHERE)[:64]
    rect = np.flatnonzero(kinds == _ffi.RT_SHAPE_RECTANGLE)[:16]
    odd = [np.array([[0, 0, 0, math.nan, 0, 1], [math.nan, 0, 0, 0, 0, 1], [1, 2, 3, 0, 0, 0], [0, 0, 0, 0, 0, 0],
                     [0, 0, 0, math.inf, 0, 0], [0, 0, -10, 0, 0, math.inf], [math.inf, 0, 0, -1, 0, 0],
                     [0, 0, -10, -math.inf, math.inf, 1]], dtype=np.float64)]
    if len(sph):
        odd.append(world_rays(d, sph, np.tile([1.0, 0.0, -10.0], (len(sph), 1)), np.tile([0.0, 0.0, 1.0], (len(sph), 1))))
    if len(rect):
        params = np.ctypeslib.as_array(d.params, shape=(n_shapes, 8))[rect]
        o = np.stack([params[:, 0] - 1.0, 0.5 * (params[:, 1] + params[:, 3]), np.zeros(len(rect))], 1)
        odd.append(world_rays(d, rect, o, np.tile([1.0, 0.0, 0.0], (len(rect), 1))))
    out["edges"] = (np.concatenate(odd), 0.001, math.inf)
    return out


def bound_edges(sc, rays, t_min, rng):
    """per-ray bounds at the decision edges: BRUTE's own hit t, one double below and above it, t_min and one double below
    it, 0, -0, negative, +inf and NaN -- one of them per ray"""
    t = nearest(sc, rays, t_min, math.inf)
    ht = np.where(t["index"] >= 0, t["t"], 1.0)
    choices = np.stack([ht, np.nextafter(ht, -np.inf), np.nextafter(ht, np.inf), np.full_like(ht, t_min),
                        np.full_like(ht, np.nextafter(t_min, -np.inf)), np.zeros_like(ht), np.full_like(ht, -0.0),
                        np.full_like(ht, -2.5), np.full_like(ht, np.inf), np.full_like(ht, np.nan)], 1)
    return np.ascontiguousarray(choices[np.arange(len(rays)), rng.integers(0, choices.shape[1], len(rays))])


@pytest.mark.parametrize("name", SCENES)
def test_scenes_and_ray_sets(name):
    sc, cam, torus = load(name)
    sets = ray_sets(sc, cam, seed=len(name))
    if name == "degenerate":
        sets["degenerate"] = (DEGENERATE_RAYS, 0.001, math.inf)
    osc = None if torus else po.OracleScene(sc.desc())
    for what, (rays, t_min, t_max) in sets.items():
        want = assert_occluded(sc, rays, t_min, t_max)
        if what in ("camera", "cfg2"):
            assert want.any()
        if osc is not None:
            sub = slice(0, 256)
            tm = t_max if np.isscalar(t_max) else t_max[sub]
            if np.isscalar(tm):
                ref = osc.intersect_batch(rays[sub], t_min, tm)["index"] >= 0
            else:
                ref = np.array([osc.intersect_batch(rays[k:k + 1], t_min, tm[k])["index"][0] >= 0
                                for k in range(len(tm))], bool)
            assert np.array_equal(want[sub], ref), f"{what}: the device's literal loop differs from the oracle"
    if name == "degenerate":
        occ = sc.occluded(DEGENERATE_RAYS, mode=rt.RT_ISECT_FAST)
        assert occ[:5].all()   # the D == 0 hits (one at t = -10), the hit at t_min and the NaN t all occlude


@pytest.mark.parametrize("name", SCENES)
def test_interval_edges_per_ray(name):
    sc, cam, _ = load(name)
    rng = np.random.default_rng(7)
    sets = ray_sets(sc, cam, seed=3)
    rays = np.concatenate([sets[k][0] for k in ("cfg2", "camera", "inside", "axes", "edges")])[:1500]
    rays = np.ascontiguousarray(rays)
    tmax = bound_edges(sc, rays, 0.001, rng)
    assert_occluded(sc, rays, 0.001, tmax)
    # the hit t itself is occluded (t == max_t is accepted), one double below it is not for a non-degenerate hit
    t = nearest(sc, rays, 0.001, math.inf)
    hit = (t["index"] >= 0) & np.isfinite(t["t"])
    assert sc.occluded(rays[hit], 0.001, np.ascontiguousarray(t["t"][hit])).all()
    for edge in (0.0, -0.0, -1.0, math.inf, math.nan, 0.001, np.nextafter(0.001, -1.0)):
        assert_occluded(sc, rays, 0.001, edge)


def test_sizes():
    sc, cam, _ = load("cornell_box.json")
    rays = np.ascontiguousarray(np.concatenate([ray_sets(sc, cam, 1)["camera"][0], bench_rays(1 << 12, seed=2)]))
    for n in (1, 255, 257):
        assert_occluded(sc, rays[:n])
        assert_occluded(sc, rays[:n], t_max=np.ascontiguousarray(np.linspace(0.5, 2000.0, n)))
    n = (1 << 20) + 3
    big = np.ascontiguousarray(np.concatenate([bench_rays(n - len(rays), seed=4), rays]))
    tmax = np.ascontiguousarray(np.array([3.0, 11.0, 700.0, math.inf])[np.arange(n) % 4])
    assert_occluded(sc, big)
    assert_occluded(sc, big, t_max=tmax, modes=(rt.RT_ISECT_FAST, rt.RT_ISECT_VERIFY))
    assert sc.occluded(np.zeros((0, 6))).shape == (0,)


def test_invalid_arguments_on_a_live_handle():
    sc, _, _ = load("cube_test.json")
    h = sc.device_scene(0)
    lib = _ffi.core()
    rays = np.ascontiguousarray(bench_rays(8))
    occ = np.zeros(8, np.uint8)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    assert lib.rt_occluded_batch(h, p(rays), 8, 0.001, math.inf, None, 3, p(occ)) == _ffi.RT_ERR_INVALID
    assert lib.rt_occluded_batch(h, p(rays), 0, 0.001, math.inf, None, -1, p(occ)) == _ffi.RT_ERR_INVALID
    assert lib.rt_occluded_batch(h, None, 8, 0.001, math.inf, None, rt.RT_ISECT_FAST, p(occ)) == _ffi.RT_ERR_INVALID
    assert lib.rt_occluded_batch(h, p(rays), 8, 0.001, math.inf, None, rt.RT_ISECT_FAST, None) == _ffi.RT_ERR_INVALID
    assert lib.rt_occluded_batch(h, None, 0, 0.001, math.inf, None, rt.RT_ISECT_FAST, None) == _ffi.RT_OK
    assert lib.rt_occluded_batch_device(h, None, 8, 0.001, math.inf, None, rt.RT_ISECT_FAST, None, None) == \
        _ffi.RT_ERR_INVALID
    assert lib.rt_occluded_batch_device(h, None, 0, 0.001, math.inf, None, rt.RT_ISECT_FAST, None, None) == _ffi.RT_OK
    with pytest.raises(ValueError):
        sc.occluded(rays, max_t=np.ones(7))


def test_device_form_on_a_torch_stream():
    torch = pytest.importorskip("torch")
    sc, cam, _ = load("dupin.json")
    sets = ray_sets(sc, cam, seed=5)
    rays, _, tmax = sets["shadow"]
    rays = np.ascontiguousarray(np.concatenate([rays, sets["camera"][0]]))
    tmax = np.ascontiguousarray(np.concatenate([tmax, np.full(len(sets["camera"][0]), 9.0)]))
    h = sc.device_scene(0)
    d_rays = torch.from_numpy(rays).cuda()
    d_tmax = torch.from_numpy(tmax).cuda()
    s = torch.cuda.Stream()
    for mode in MODES:
        out_s = torch.empty(len(rays), dtype=torch.uint8, device="cuda")
        out_v = torch.empty(len(rays), dtype=torch.bool, device="cuda")
        with torch.cuda.stream(s):
            api.occluded_device(h, d_rays, out_s, t_max=7.5, mode=mode)
            api.occluded_device(h, d_rays, out_v, t_max=d_tmax, mode=mode)
        s.synchronize()
        assert np.array_equal(out_s.cpu().numpy().astype(bool), sc.occluded(rays, 0.001, 7.5, mode=mode))
        assert np.array_equal(out_v.cpu().numpy(), sc.occluded(rays, 0.001, tmax, mode=mode))
    # the default stream (cudaStreamLegacy)
    out = torch.empty(len(rays), dtype=torch.uint8, device="cuda")
    api.occluded_device(h, d_rays, out, t_max=d_tmax)
    assert np.array_equal(out.cpu().numpy().astype(bool), reference(sc, rays, 0.001, tmax))
    with pytest.raises(ValueError):
        api.occluded_device(h, d_rays, out, t_max=d_tmax[::2])
    with pytest.raises(ValueError):
        api.occluded_device(h, d_rays, out[:-1])


def test_multi_device_handle_answers_on_its_first_device():
    sc, cam, _ = load("cornell_box.json")
    rays, _, tmax = ray_sets(sc, cam, seed=9)["shadow"]
    rays = np.ascontiguousarray(rays)
    want = reference(sc, rays, 0.001, tmax)
    hm = sc.device_scene_multi(list(range(rt.device_count())))
    out = np.empty(len(rays), np.uint8)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    for mode in MODES:
        assert _ffi.core().rt_occluded_batch(hm, p(rays), len(rays), 0.001, math.inf, p(tmax), mode, p(out)) == 0
        assert np.array_equal(out.astype(bool), want)


def _occluded_h(h, rays, tmax, mode):
    out = np.empty(len(rays), np.uint8)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    assert _ffi.core().rt_occluded_batch(h, p(rays), len(rays), 0.001, math.inf, p(tmax), mode, p(out)) == 0, \
        _ffi.core().rt_last_error()
    return out


@pytest.mark.parametrize("name", ["spheres.json", "dupin.json", "big"])
def test_scene_updates(name):
    sc, cam, _ = load(name)
    ed = Edited(sc)
    rng = np.random.default_rng(4)
    sets = ray_sets(sc, cam, seed=2)
    rays = np.ascontiguousarray(np.concatenate([sets["camera"][0], sets["cfg2"][0], sets["shadow"][0]]))
    tmax = np.ascontiguousarray(np.concatenate([np.full(len(rays) - len(sets["shadow"][0]), np.inf), sets["shadow"][2]]))
    h = create(ed.desc())
    try:
        before = _occluded_h(h, rays, tmax, rt.RT_ISECT_FAST)
        index = rng.choice(len(ed.inv), size=min(len(ed.inv), 100), replace=False)
        update_transforms(h, index, *ed.move(rng, index, 1.0))
        fresh = create(ed.desc())
        try:
            for mode in MODES:
                assert np.array_equal(_occluded_h(h, rays, tmax, mode), _occluded_h(fresh, rays, tmax, mode))
        finally:
            _ffi.core().rt_scene_destroy(fresh)
        assert not np.array_equal(_occluded_h(h, rays, tmax, rt.RT_ISECT_FAST), before)
        other, _, _ = load("cornell_box.json")
        api.scene_update(h, other.desc())
        fresh = create(other.desc())
        try:
            for mode in MODES:
                assert np.array_equal(_occluded_h(h, rays, tmax, mode), _occluded_h(fresh, rays, tmax, mode))
        finally:
            _ffi.core().rt_scene_destroy(fresh)
    finally:
        _ffi.core().rt_scene_destroy(h)


def test_device_queries_are_ordered_against_updates():
    """rt_occluded_batch_device queued on a torch stream before an update sees the old scene, after it the new one"""
    torch = pytest.importorskip("torch")
    sc, cam, _ = load("spheres.json")
    ed = Edited(sc)
    rng = np.random.default_rng(11)
    rays = np.ascontiguousarray(np.concatenate([ray_sets(sc, cam, seed=6)["camera"][0], bench_rays(1 << 16, seed=6)]))
    tmax = np.ascontiguousarray(rng.uniform(1.0, 30.0, len(rays)))
    h = create(ed.desc())
    try:
        old = _occluded_h(h, rays, tmax, rt.RT_ISECT_FAST)
        index = np.flatnonzero(sc.shape_kinds() == _ffi.RT_SHAPE_SPHERE)[:200]
        inv, direct = ed.move(rng, index, 2.0)
        fresh = create(ed.desc())
        new = _occluded_h(fresh, rays, tmax, rt.RT_ISECT_FAST)
        _ffi.core().rt_scene_destroy(fresh)
        assert not np.array_equal(old, new)
        s = torch.cuda.Stream()
        d_rays, d_tmax = torch.from_numpy(rays).cuda(), torch.from_numpy(tmax).cuda()
        before = torch.empty(len(rays), dtype=torch.uint8, device="cuda")
        after = torch.empty_like(before)
        with torch.cuda.stream(s):
            for _ in range(8):   # enough work queued that the update would overtake it if it were not ordered
                api.occluded_device(h, d_rays, before, t_max=d_tmax, mode=rt.RT_ISECT_BRUTE)
            update_transforms(h, index, inv, direct)
            api.occluded_device(h, d_rays, after, t_max=d_tmax, mode=rt.RT_ISECT_FAST)
        s.synchronize()
        assert np.array_equal(before.cpu().numpy(), old)
        assert np.array_equal(after.cpu().numpy(), new)
    finally:
        _ffi.core().rt_scene_destroy(h)


@pytest.mark.parametrize("name", ["cornell_box.json", "dupin.json", "big"])
def test_counters_show_the_early_exit(name):
    sc, cam, _ = load(name)
    rays, t_min, tmax = ray_sets(sc, cam, seed=8)["shadow"]
    rays = np.ascontiguousarray(rays)
    occ = reference(sc, rays, t_min, tmax)
    assert occ.sum() > 20
    blocked, free = rays[occ], rays[~occ]
    sc.set_counters(True)
    try:
        for mode in (rt.RT_ISECT_BRUTE, rt.RT_ISECT_FAST):
            sc.reset_stats()
            assert sc.occluded(blocked, t_min, np.ascontiguousarray(tmax[occ]), mode=mode).all()
            st = sc.stats()
            assert st.segments == len(blocked)
            any_tests = st.shape_tests
            sc.reset_stats()
            sc.closest_hit(blocked, t_min, math.inf, mode=mode, want=("index",))
            assert sc.stats().segments == len(blocked)
            assert any_tests < sc.stats().shape_tests, (mode, any_tests, sc.stats().shape_tests)
        sc.reset_stats()
        sc.occluded(free, t_min, np.ascontiguousarray(tmax[~occ]), mode=rt.RT_ISECT_FAST)
        assert sc.stats().segments == len(free)
        ms = sc.stats().last_intersect_ms
        sc.occluded(free, t_min, 1.0)
        assert sc.stats().last_intersect_ms == ms   # not touched
    finally:
        sc.set_counters(False)


def test_kernel_timing_does_not_change_answers():
    sc, cam, _ = load("dupin.json")
    rays, t_min, tmax = ray_sets(sc, cam, seed=12)["shadow"]
    rays = np.ascontiguousarray(rays)
    want = [sc.occluded(rays, t_min, tmax, mode=m) for m in MODES]
    sc.set_kernel_timing(True)
    try:
        assert all(np.array_equal(sc.occluded(rays, t_min, tmax, mode=m), w) for m, w in zip(MODES, want))
    finally:
        sc.set_kernel_timing(False)


def test_big_scene_box_rays():
    """the generated 10^4-shape scene with levels above the roots, rays from all around it"""
    sc, _, _ = load("big")
    rays = np.ascontiguousarray(box_rays(1 << 14, seed=3, extent=25.0))
    rng = np.random.default_rng(1)
    assert_occluded(sc, rays)
    assert_occluded(sc, rays, t_max=np.ascontiguousarray(rng.uniform(0.0, 60.0, len(rays))))
