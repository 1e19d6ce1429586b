"""Scatter queries (rt_scatter_batch[_device]): one segment of ray_color for caller rays, against the oracle per ray
and composed into the frame bit for bit.

Per ray, the nearest hit (index, t), the outcome and the scattered ray must be the oracle's bit for bit
(tests/oracle_scatter.cpp: collection_ray_intersect, material_scatter / material_emitted / background and the Philox
PathRng keyed as the frame keys it).  The colour is compared bit for bit wherever its texture chain evaluates no sin,
acos or atan2 (glibc's libm against CUDA's libdevice elsewhere); there the number of differing rays is printed, and the
composed paths must pass check_groups' one-float-ulp-per-path bound.

The main gate: api.trace_paths over each pixel's camera rays, averaged by api.group_means, is
rt_trace_pixel_samples_group and the rt_render_start frame bit for bit."""
import ctypes as C
import json
import math

import numpy as np
import pytest

import rs_pathtracing_b200 as rt
from rs_pathtracing_b200 import _ffi, api
from oracle import pyoracle as po

import scatter_oracle
from conftest import scene_path
from test_gpu_caller_rays import check_groups
from test_gpu_frame_edges import marched_scene
from test_gpu_intersect import bench_rays
from test_gpu_occluded import SCENES, load, ray_sets
from test_gpu_render import _variant_4b
from test_gpu_scene_update import Edited, create, update_transforms
from test_gpu_trace_group import _primary_rays

pytestmark = pytest.mark.gpu

MODES = (rt.RT_ISECT_BRUTE, rt.RT_ISECT_FAST, rt.RT_ISECT_VERIFY)
OUTPUTS = api.SCATTER_OUTPUTS
p = lambda a: a.ctypes.data_as(C.c_void_p) if a is not None else None


def random_keys(rng, n):
    """pixel / sample keys with the extremes 0 and 0xFFFFFFFF in both places"""
    keys = rng.integers(0, 1 << 32, (n, 2), dtype=np.uint64).astype(np.uint32)
    edge = np.array([[0, 0], [0xFFFFFFFF, 0xFFFFFFFF], [0, 0xFFFFFFFF], [0xFFFFFFFF, 0]], np.uint32)
    keys[:min(n, 4)] = edge[:min(n, 4)]
    return np.ascontiguousarray(keys)


def same(a, b):
    """bit for bit, NaN payloads and signed zeros included"""
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.tobytes() == b.tobytes()


def scatter_h(h, rays, keys, level, seed=0, mode=rt.RT_ISECT_FAST, want=OUTPUTS, t_min=0.001, t_max=math.inf):
    """rt_scatter_batch on a raw handle with only the outputs in `want` (the others NULL)"""
    n = len(rays)
    out = {"index": np.empty(n, np.int32), "t": np.empty(n), "outcome": np.empty(n, np.uint8),
           "color": np.empty((n, 3)), "scattered": np.empty((n, 6))}
    out = {k: (v if k in want else None) for k, v in out.items()}
    rays, keys = np.ascontiguousarray(rays, np.float64), np.ascontiguousarray(keys, np.uint32)
    rc = _ffi.core().rt_scatter_batch(h, p(rays), p(keys), n, level, seed, t_min, t_max, mode,
                                      *(p(out[k]) for k in OUTPUTS))
    assert rc == 0, _ffi.core().rt_last_error()
    return {k: v for k, v in out.items() if v is not None}


def exact_colour(sc, index):
    """rays whose colour involves no sin / acos / atan2: misses (sky), Dielectric and EmptyMaterial, a SolidColor root
    texture, and an image texture on a Cube, Rectangle or marched shape"""
    d = sc.desc()
    kinds = sc.shape_kinds()
    out = np.ones(len(index), bool)
    for k, i in enumerate(index):
        if i < 0:
            continue
        m = d.materials[d.material[i]]
        if m.kind in (_ffi.RT_MAT_DIELECTRIC, _ffi.RT_MAT_EMPTY):
            continue
        tk = d.textures[m.texture].kind
        out[k] = tk == _ffi.RT_TEX_SOLID or (tk == _ffi.RT_TEX_IMAGE and kinds[i] not in (_ffi.RT_SHAPE_SPHERE,
                                                                                           _ffi.RT_SHAPE_TORUS))
    return out


def check_against_oracle(sc, osc, rays, keys, level, seed, what):
    got = sc.scatter(rays, keys, level, seed)
    want = scatter_oracle.scatter_batch(osc, rays, keys, level, seed)
    for k in ("index", "t", "outcome", "scattered"):
        ok = (got[k] == want[k]) | (np.isnan(got[k]) & np.isnan(want[k]))
        bad = np.flatnonzero(~ok.reshape(len(rays), -1).all(1))
        assert bad.size == 0, f"{what} {k}: {bad.size} of {len(rays)} differ, first ray {rays[bad[0]].tolist()}"
    exact = exact_colour(sc, want["index"])
    eq = (got["color"] == want["color"]) | (np.isnan(got["color"]) & np.isnan(want["color"]))
    assert eq[exact].all(), f"{what} color: {int((~eq[exact]).any(1).sum())} exact rays differ"
    print(f"{what}: {int((~eq[~exact]).any(1).sum())} of {int((~exact).sum())} libm-chain colours differ")
    # unused outputs are zero
    oc = got["outcome"]
    assert (got["index"][oc == rt.RT_BOUNCE_MISS] == -1).all() and (got["t"][oc == rt.RT_BOUNCE_MISS] == 0).all()
    assert (got["scattered"][oc != rt.RT_BOUNCE_SCATTER] == 0).all()
    return got


@pytest.mark.parametrize("name", [s for s in SCENES if s != "torus.json"])
def test_against_the_oracle_per_ray(name):
    sc, cam, _ = load(name)
    osc = po.OracleScene(sc.desc())
    rng = np.random.default_rng(len(name))
    for what, (rays, _, _) in ray_sets(sc, cam, seed=len(name)).items():
        rays = np.ascontiguousarray(rays[:1024])
        keys = random_keys(rng, len(rays))
        for level in (0, 5):
            check_against_oracle(sc, osc, rays, keys, level, (1 << 64) - 1 if level else 0, f"{name} {what} {level}")


def test_torus_against_the_oracle():
    """the Torus's quartic takes glibc's and CUDA's libm: compared as tests/test_torus.py compares its nearest hit"""
    sc, cam, _ = load("torus.json")
    osc = po.OracleScene(sc.desc())
    w, h = 160, 120
    rays = np.array([po.get_ray(cam, w, h, x + 0.5, y + 0.5) for y in range(h) for x in range(w)])
    keys = random_keys(np.random.default_rng(2), len(rays))
    got = sc.scatter(rays, keys, 1, 9)
    want = scatter_oracle.scatter_batch(osc, rays, keys, 1, 9)
    d = sc.desc()
    tor = [i for i in range(d.n_shapes) if int(d.kind[i]) == _ffi.RT_SHAPE_TORUS]
    on_torus = np.isin(want["index"], tor) | np.isin(got["index"], tor)
    assert on_torus.sum() > 1500
    agree = got["index"] == want["index"]
    assert agree[~on_torus].all()
    off = ~on_torus
    for k in ("t", "outcome", "scattered"):
        assert np.array_equal(got[k][off], want[k][off]), k
    hit = agree & (want["index"] >= 0)
    rel = np.zeros(len(rays))
    rel[hit] = np.abs(got["t"][hit] - want["t"][hit]) / np.abs(want["t"][hit])
    differs = on_torus & (~agree | (rel > 1e-9))
    assert differs.sum() <= 0.03 * on_torus.sum(), (differs.sum(), on_torus.sum())
    ok = on_torus & ~differs
    assert (got["outcome"][ok] == want["outcome"][ok]).all()
    s = ok & (want["outcome"] == rt.RT_BOUNCE_SCATTER)
    assert np.abs(got["scattered"][s] - want["scattered"][s]).max() < 1e-6


def test_modes_agree_and_verify_is_clean():
    for name in ("cornell_box.json", "dupin.json", "4b", "big"):
        sc, cam, _ = load(name)
        sets = ray_sets(sc, cam, seed=4)
        rays = np.ascontiguousarray(np.concatenate([sets[k][0] for k in ("camera", "secondary", "inside", "edges")]))
        keys = random_keys(np.random.default_rng(1), len(rays))
        ref = None
        for mode in MODES:
            sc.reset_stats()
            got = sc.scatter(rays, keys, 3, 17, mode=mode)
            if mode == rt.RT_ISECT_VERIFY:
                st = sc.stats()
                assert (st.verify_rays, st.verify_false_culls) == (0, 0), name
            if ref is None:
                ref = got
            assert all(same(got[k], ref[k]) for k in OUTPUTS), (name, mode)
        hit = sc.closest_hit(rays, mode=rt.RT_ISECT_BRUTE, want=("index", "t"))
        assert same(ref["index"], hit["index"]) and same(ref["t"], hit["t"])


def test_each_output_alone():
    sc, cam, _ = load("4b")
    h = sc.device_scene(0)
    sets = ray_sets(sc, cam, seed=6)
    rays = np.ascontiguousarray(np.concatenate([sets["camera"][0], sets["secondary"][0]]))
    keys = random_keys(np.random.default_rng(6), len(rays))
    full = scatter_h(h, rays, keys, 2, 5)
    for k in OUTPUTS:
        assert same(scatter_h(h, rays, keys, 2, 5, want=(k,))[k], full[k]), k
    assert scatter_h(h, rays, keys, 2, 5, want=()) == {}
    # the device form with only its two required outputs, then each other output with them
    torch = pytest.importorskip("torch")
    d_rays, d_keys = torch.from_numpy(rays).cuda(), torch.from_numpy(keys.view(np.int32)).cuda()
    n = len(rays)
    for extra in (None, "outcome", "color", "scattered"):
        outs = {"index": torch.empty(n, dtype=torch.int32, device="cuda"),
                "t": torch.empty(n, dtype=torch.float64, device="cuda"),
                "outcome": torch.empty(n, dtype=torch.uint8, device="cuda") if extra == "outcome" else None,
                "color": torch.empty((n, 3), dtype=torch.float64, device="cuda") if extra == "color" else None,
                "scattered": torch.empty((n, 6), dtype=torch.float64, device="cuda") if extra == "scattered" else None}
        rc = _ffi.core().rt_scatter_batch_device(h, d_rays.data_ptr(), d_keys.data_ptr(), n, 2, 5, 0.001, math.inf,
                                                 rt.RT_ISECT_FAST,
                                                 *((outs[k].data_ptr() if outs[k] is not None else None) for k in OUTPUTS),
                                                 None)
        assert rc == 0, _ffi.core().rt_last_error()
        torch.cuda.synchronize()
        for k, v in outs.items():
            if v is not None:
                assert same(v.cpu().numpy(), full[k]), (extra, k)


def test_invalid_arguments_on_a_live_handle():
    sc, _, _ = load("cube_test.json")
    h = sc.device_scene(0)
    lib = _ffi.core()
    rays = np.ascontiguousarray(bench_rays(8))
    keys = np.zeros((8, 2), np.uint32)
    outs = [np.empty(8, np.int32), np.empty(8), np.empty(8, np.uint8), np.empty((8, 3)), np.empty((8, 6))]
    F = rt.RT_ISECT_FAST
    for fn, extra in ((lib.rt_scatter_batch, ()), (lib.rt_scatter_batch_device, (None,))):
        call = lambda r, k, n, level, mode, o=outs: fn(h, r, k, n, level, 0, 0.001, math.inf, mode, *map(p, o), *extra)
        assert call(None, None, 0, 63, 3) == _ffi.RT_ERR_INVALID and b"mode" in lib.rt_last_error()
        assert call(None, None, 0, 63, F) == _ffi.RT_ERR_INVALID and b"level" in lib.rt_last_error()
        assert call(None, p(keys), 8, 0, F) == _ffi.RT_ERR_INVALID and b"rays" in lib.rt_last_error()
        assert call(p(rays), None, 8, 0, F) == _ffi.RT_ERR_INVALID and b"keys" in lib.rt_last_error()
        assert call(None, None, 0, 62, F) == _ffi.RT_OK
    # the device form needs its index and t buffers; the host form takes NULL for every output
    nulls = [None] * 5
    assert lib.rt_scatter_batch_device(h, p(rays), p(keys), 8, 0, 0, 0.001, math.inf, F, *nulls, None) == \
        _ffi.RT_ERR_INVALID
    assert lib.rt_scatter_batch(h, p(rays), p(keys), 8, 0, 0, 0.001, math.inf, F, *nulls) == _ffi.RT_OK
    for level in (0, 62):
        assert sc.scatter(rays, keys, level)["index"].shape == (8,)
    with pytest.raises(rt.RtError, match="level"):
        sc.scatter(rays, keys, 63)
    assert sc.scatter(np.zeros((0, 6)), np.zeros((0, 2), np.uint32), 0)["color"].shape == (0, 3)


def test_sizes_and_keys():
    sc, cam, _ = load("cornell_box.json")
    osc = po.OracleScene(sc.desc())
    base = np.ascontiguousarray(np.concatenate([ray_sets(sc, cam, 1)["camera"][0], bench_rays(1 << 12, seed=2)]))
    rng = np.random.default_rng(3)
    for n in (1, 255, 257):
        check_against_oracle(sc, osc, base[:n], random_keys(rng, n), 1, 11, f"n={n}")
    n = (1 << 20) + 3
    big = np.ascontiguousarray(np.concatenate([bench_rays(n - len(base), seed=4), base]))
    keys = random_keys(rng, n)
    got = sc.scatter(big, keys, 1, 11)
    sub = rng.choice(n, 4096, replace=False)
    sub[:3] = [0, n - 2, n - 1]
    want = scatter_oracle.scatter_batch(osc, big[sub], keys[sub], 1, 11)
    for k in ("index", "t", "outcome", "scattered"):
        assert same(got[k][sub], want[k]), k
    # repeated (ray, key) pairs give repeated answers, wherever they sit in the batch; a different key another sample
    rep = np.ascontiguousarray(np.repeat(base[:64], 5, axis=0))
    rkeys = np.ascontiguousarray(np.repeat(random_keys(rng, 64), 5, axis=0))
    got = sc.scatter(rep, rkeys, 0, 2)
    for k in OUTPUTS:
        a = got[k].reshape(64, 5, -1)
        assert (a == a[:, :1]).all(), k
    other = rkeys.copy()
    other[:, 1] ^= 1
    diffuse = got["outcome"] == rt.RT_BOUNCE_SCATTER
    assert not same(sc.scatter(rep, other, 0, 2)["scattered"][diffuse], got["scattered"][diffuse])


COMPOSE = ["spheres.json", "cornell_box.json", "dupin.json", "4b", "light_source.json", "march33"]


def _compose_scene(name):
    if name == "march33":   # 33 ray-marched shapes: the group entry runs the fused k_bounce
        sc = rt.Scene.from_json(json.dumps(marched_scene(33)), add_random_spheres=False)
        return sc, sc.camera()
    if name == "4b":
        sc = rt.Scene.from_file(scene_path("detached_materials.json"), random_spheres_seed=1)
        return sc, _variant_4b(sc)
    sc = rt.Scene.from_file(scene_path(name), random_spheres_seed=1)
    return sc, sc.camera()


@pytest.mark.parametrize("name", COMPOSE)
def test_trace_paths_reproduces_the_group_entry_and_the_frame(name):
    torch = pytest.importorskip("torch")
    w, h, spp = 20, 14, 3
    sc, cam = _compose_scene(name)
    pix = np.arange(w * h, dtype=np.uint32)
    offsets = np.arange(0, w * h * spp + 1, spp, dtype=np.uint64)
    keys = np.ascontiguousarray(np.stack([np.repeat(pix, spp), np.tile(np.arange(spp, dtype=np.uint32), w * h)], 1))
    for seed in (0, (1 << 64) - 1):
        rays = np.ascontiguousarray(_primary_rays(cam, w, h, spp, seed))
        for depth in (0, 1, 8, 62):
            if seed:   # the torch path: every level on torch's current stream
                L = api.trace_paths(sc, torch.from_numpy(rays).cuda(), torch.from_numpy(keys.view(np.int32)).cuda()
                                    .view(torch.uint32), depth, seed)
                assert L.dtype == torch.float32 and L.is_cuda
            else:
                L = api.trace_paths(sc, rays, keys, depth, seed)
                assert L.dtype == np.float32
            got = api.group_means(L, offsets)
            group = sc.trace_pixel_samples_group(rays, offsets, pix, depth, seed=seed)
            assert same(got, group), (name, seed, depth)
            frame = rt.GpuRenderer(sc, 12, depth, seed=seed).render(cam, w, h, spp)
            assert same(got, frame.reshape(-1, 3)), (name, seed, depth)
            if depth == 8 and name != "march33":
                osc = po.OracleScene(sc.desc())
                cols = osc.group_sample_colors(rays, offsets, pix, depth, seed)
                check_groups(got, cols, offsets, f"{name} trace_paths seed {seed}")


def test_record_holds_each_level():
    sc, cam = _compose_scene("cornell_box.json")
    w, h, spp, depth, seed = 8, 6, 4, 6, 21
    rays = np.ascontiguousarray(_primary_rays(cam, w, h, spp, seed))
    keys = np.ascontiguousarray(np.stack([np.repeat(np.arange(w * h, dtype=np.uint32), spp),
                                          np.tile(np.arange(spp, dtype=np.uint32), w * h)], 1))
    L, levels = api.trace_paths(sc, rays, keys, depth, seed, record=True)
    assert same(L, api.trace_paths(sc, rays, keys, depth, seed))
    assert 1 <= len(levels) <= depth + 1 and same(levels[0]["ray"], np.arange(len(rays)))
    for k, v in enumerate(levels):
        assert len(v["ray"]) == len(v["shape"]) == len(v["outcome"]) == len(v["color"]) == len(v["beta"])
        if k + 1 < len(levels):
            nxt = levels[k + 1]
            go = v["outcome"] == rt.RT_BOUNCE_SCATTER
            assert same(nxt["ray"], v["ray"][go])
            assert same(nxt["beta"], v["beta"][go] * v["color"][go])


def test_device_form_matches_the_host_form():
    torch = pytest.importorskip("torch")
    sc, cam, _ = load("dupin.json")
    sets = ray_sets(sc, cam, seed=5)
    rays = np.ascontiguousarray(np.concatenate([sets["camera"][0], sets["secondary"][0], sets["edges"][0]]))
    keys = random_keys(np.random.default_rng(5), len(rays))
    d_rays = torch.from_numpy(rays).cuda()
    d_keys = torch.from_numpy(keys.view(np.int32)).cuda().view(torch.uint32)
    s = torch.cuda.Stream()
    for mode in MODES:
        want = sc.scatter(rays, keys, 4, 8, mode=mode)
        with torch.cuda.stream(s):
            got = sc.scatter(d_rays, d_keys, 4, 8, mode=mode)
        s.synchronize()
        assert all(same(got[k].cpu().numpy(), want[k]) for k in OUTPUTS), mode
    got = sc.scatter(d_rays, d_keys, 4, 8)   # the default stream (cudaStreamLegacy)
    torch.cuda.synchronize()
    want = sc.scatter(rays, keys, 4, 8)
    assert all(same(got[k].cpu().numpy(), want[k]) for k in OUTPUTS)
    with pytest.raises(ValueError):
        sc.scatter(d_rays, d_keys[:-1], 0)
    with pytest.raises(ValueError):
        sc.scatter(d_rays[:, :3], d_keys, 0)


@pytest.mark.parametrize("name", ["spheres.json", "dupin.json", "big"])
def test_scene_updates(name):
    """after a transforms update and after a full update the handle answers as a fresh handle of the edited scene"""
    sc, cam, _ = load(name)
    ed = Edited(sc)
    rng = np.random.default_rng(4)
    sets = ray_sets(sc, cam, seed=2)
    rays = np.ascontiguousarray(np.concatenate([sets["camera"][0], sets["secondary"][0], sets["cfg2"][0]]))
    keys = random_keys(rng, len(rays))
    h = create(ed.desc())

    def same_as_fresh(desc):
        fresh = create(desc)
        try:
            for mode in MODES:
                a, b = scatter_h(h, rays, keys, 1, 3, mode=mode), scatter_h(fresh, rays, keys, 1, 3, mode=mode)
                assert all(same(a[k], b[k]) for k in OUTPUTS), (name, mode)
        finally:
            _ffi.core().rt_scene_destroy(fresh)

    try:
        before = scatter_h(h, rays, keys, 1, 3)
        index = rng.choice(len(ed.inv), size=min(len(ed.inv), 100), replace=False)
        update_transforms(h, index, *ed.move(rng, index, 1.0))
        same_as_fresh(ed.desc())
        assert not same(scatter_h(h, rays, keys, 1, 3)["color"], before["color"])
        other, _, _ = load("cornell_box.json")
        api.scene_update(h, other.desc())
        same_as_fresh(other.desc())
    finally:
        _ffi.core().rt_scene_destroy(h)


def test_device_queries_are_ordered_against_updates():
    """rt_scatter_batch_device queued on a torch stream before an update sees the old scene, after it the new one"""
    torch = pytest.importorskip("torch")
    sc, cam, _ = load("spheres.json")
    ed = Edited(sc)
    rng = np.random.default_rng(11)
    rays = np.ascontiguousarray(np.concatenate([ray_sets(sc, cam, seed=6)["camera"][0], bench_rays(1 << 16, seed=6)]))
    keys = random_keys(rng, len(rays))
    h = create(ed.desc())
    n = len(rays)
    try:
        old = scatter_h(h, rays, keys, 2, 1)
        index = np.flatnonzero(sc.shape_kinds() == _ffi.RT_SHAPE_SPHERE)[:200]
        inv, direct = ed.move(rng, index, 2.0)
        fresh = create(ed.desc())
        new = scatter_h(fresh, rays, keys, 2, 1)
        _ffi.core().rt_scene_destroy(fresh)
        assert not same(old["color"], new["color"])
        s = torch.cuda.Stream()
        d_rays = torch.from_numpy(rays).cuda()
        d_keys = torch.from_numpy(keys.view(np.int32)).cuda()
        bufs = lambda: {"index": torch.empty(n, dtype=torch.int32, device="cuda"),
                        "t": torch.empty(n, dtype=torch.float64, device="cuda"),
                        "outcome": torch.empty(n, dtype=torch.uint8, device="cuda"),
                        "color": torch.empty((n, 3), dtype=torch.float64, device="cuda"),
                        "scattered": torch.empty((n, 6), dtype=torch.float64, device="cuda")}
        before, after = bufs(), bufs()

        def launch(out, mode):
            rc = _ffi.core().rt_scatter_batch_device(h, d_rays.data_ptr(), d_keys.data_ptr(), n, 2, 1, 0.001, math.inf,
                                                     mode, *(out[k].data_ptr() for k in OUTPUTS), s.cuda_stream)
            assert rc == 0, _ffi.core().rt_last_error()

        with torch.cuda.stream(s):
            for _ in range(8):   # enough work queued that the update would overtake it if it were not ordered
                launch(before, rt.RT_ISECT_BRUTE)
            update_transforms(h, index, inv, direct)
            launch(after, rt.RT_ISECT_FAST)
        s.synchronize()
        assert all(same(before[k].cpu().numpy(), old[k]) for k in OUTPUTS)
        assert all(same(after[k].cpu().numpy(), new[k]) for k in OUTPUTS)
    finally:
        _ffi.core().rt_scene_destroy(h)


def test_multi_device_handle_answers_on_its_first_device():
    sc, cam, _ = load("cornell_box.json")
    rays = np.ascontiguousarray(ray_sets(sc, cam, seed=9)["secondary"][0])
    keys = random_keys(np.random.default_rng(9), len(rays))
    want = sc.scatter(rays, keys, 1, 4)
    hm = sc.device_scene_multi(list(range(rt.device_count())))
    for mode in MODES:
        got = scatter_h(hm, rays, keys, 1, 4, mode=mode)
        assert all(same(got[k], want[k]) for k in OUTPUTS), mode


def test_a_frame_in_flight_is_left_alone():
    sc, cam, _ = load("dupin.json")
    h = sc.device_scene(0)
    params = api.render_params(160, 120, 4, 8, 5)
    api.render_start(h, cam, params)
    ref = np.empty((120, 160, 3))
    api.render_wait(h, ref)
    rays = np.ascontiguousarray(ray_sets(sc, cam, seed=3)["camera"][0])
    keys = random_keys(np.random.default_rng(3), len(rays))
    want = sc.scatter(rays, keys, 2, 6)
    sc.reset_stats()
    ms = sc.stats().last_intersect_ms
    api.render_start(h, cam, params)
    got = sc.scatter(rays, keys, 2, 6)   # while the frame is in flight
    buf = np.empty((120, 160, 3))
    api.render_wait(h, buf)
    assert same(buf, ref)
    assert all(same(got[k], want[k]) for k in OUTPUTS)
    assert sc.stats().paths == 160 * 120 * 4 and sc.stats().last_intersect_ms == ms


@pytest.mark.parametrize("name", ["cornell_box.json", "dupin.json", "big"])
def test_counters_are_the_nearest_hits(name):
    sc, cam, _ = load(name)
    sets = ray_sets(sc, cam, seed=8)
    rays = np.ascontiguousarray(np.concatenate([sets["camera"][0], sets["secondary"][0]]))
    keys = random_keys(np.random.default_rng(8), len(rays))
    fields = ("segments", "shape_tests", "cull_tests", "march_steps", "march_rays", "march_long_rays")
    sc.set_counters(True)
    try:
        for mode in (rt.RT_ISECT_BRUTE, rt.RT_ISECT_FAST):
            sc.reset_stats()
            sc.scatter(rays, keys, 1, 2, mode=mode)
            a = sc.stats()
            sc.reset_stats()
            sc.closest_hit(rays, mode=mode, want=("index", "t"))
            b = sc.stats()
            assert [getattr(a, f) for f in fields] == [getattr(b, f) for f in fields], (name, mode)
            assert a.segments == len(rays)
    finally:
        sc.set_counters(False)
    want = sc.scatter(rays, keys, 1, 2)
    sc.set_kernel_timing(True)
    try:
        got = sc.scatter(rays, keys, 1, 2)
        assert all(same(got[k], want[k]) for k in OUTPUTS)
    finally:
        sc.set_kernel_timing(False)
