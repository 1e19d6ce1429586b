"""Frames against the oracle at float precision, and at the edges of depth, seed, image, tiling and batching.

The strict comparison (check_pixels).  Every path's radiance is computed in FP64 and rounded to float once; a pixel is
the f64 sum of its float samples in sample order, divided by the sample count.  So, with c_s the oracle's FP64 colour of
sample s and f_s = float32(c_s) widened back to f64, the GPU pixel G is compared with the emulated pixel
    E = (sum of f_s in sample order, from 0.0) / n
and must satisfy |G - E| <= (sum of ulp32(f_s)) / n + n * ulp64(E): each path may be off by one float ulp, never by
more.  One sample: G is f_0 or one of its two float neighbours.  The old frame tolerance (1e-7 * max(pixel, 1) * spp)
allowed a relative error of 4e-5 on a pixel of 0.01 at 4 spp; this bound allows one float ulp per path.
The number of pixels that are not bit-identical to E is printed by every check."""
import ctypes as C
import json

import numpy as np
import pytest

import rs_pathtracing_b200 as rt
from rs_pathtracing_b200 import _ffi, api
from oracle import pyoracle as po

from conftest import scene_path
from test_gpu_intersect import SURFACES, _compare, scene_rays
from test_gpu_trace_group import _primary_rays

pytestmark = pytest.mark.gpu

SEEDS = [0, (1 << 32) - 1, 1 << 32, (1 << 63) + 12345, (1 << 64) - 1]


def check_pixels(got, cols, what=""):
    """got: GPU pixels (..., 3); cols: the oracle's per-sample colours (P, n, 3) of the same pixels, all n samples in
    sample order.  Asserts the strict bound; returns the number of pixels not bit-identical to the emulated pixel."""
    got = np.asarray(got, dtype=np.float64).reshape(-1, 3)
    cols = np.asarray(cols, dtype=np.float64)
    assert got.shape[0] == cols.shape[0]
    n = cols.shape[1]
    f32 = cols.astype(np.float32)
    f = f32.astype(np.float64)
    s = np.zeros(got.shape)
    for k in range(n):
        s = s + f[:, k]
    emu = s / n
    assert np.isfinite(got).all() and np.isfinite(emu).all(), what
    if n == 1:
        f0 = f32[:, 0]
        ok = ((got == emu) | (got == np.nextafter(f0, np.float32(-np.inf)).astype(np.float64))
              | (got == np.nextafter(f0, np.float32(np.inf)).astype(np.float64)))
        bound = np.spacing(np.abs(f0)).astype(np.float64)
    else:
        bound = np.spacing(np.abs(f32)).astype(np.float64).sum(axis=1) / n + n * np.spacing(np.abs(emu))
        ok = np.abs(got - emu) <= bound
    bad = ~ok.all(axis=1)
    if bad.any():
        i = int(np.flatnonzero(bad)[0])
        raise AssertionError(f"{what}: {int(bad.sum())} of {len(got)} pixels exceed one float ulp per path; first: pixel row "
                             f"{i}, gpu {got[i].tolist()}, emulated {emu[i].tolist()}, bound {bound[i].tolist()}")
    n_diff = int((got != emu).any(axis=1).sum())
    print(f"strict-bound {what}: {n_diff} of {len(got)} pixels not bit-identical")
    return n_diff


def check_frame(got, osc, cam, w, h, spp, depth, seed, what=""):
    """a whole (h, w, 3) GPU frame against the oracle's samples 0 .. spp-1 of every pixel"""
    return check_pixels(got, osc.frame_sample_colors(cam, w, h, spp, depth, seed), what)


# ---- helpers -----------------------------------------------------------------------------------------------------

def _core():
    return _ffi.core()


def _params(w, h, spp, depth, seed, shards=1, index=0, tile=(0, 0)):
    p = api.render_params(w, h, spp, depth, seed, shards, index)
    p.tile_width, p.tile_height = tile
    return p


def _load(name):
    if name in MARCH_SCENES:
        return rt.Scene.from_json(json.dumps(marched_scene(MARCH_SCENES[name])), add_random_spheres=False)
    return rt.Scene.from_file(scene_path(name), random_spheres_seed=1)


def _frame(sc, cam, w, h, spp, depth, seed):
    return rt.GpuRenderer(sc, 12, depth, seed=seed).render(cam, w, h, spp)


def _poll_frame(handle, cam, params, buf):
    """rt_render_start, then rt_render_poll until done: partial ranges of batches are delivered as they finish"""
    api.render_start(handle, cam, params)
    polls = 0
    while not api.render_poll(handle, buf):
        polls += 1
    return polls


def _adaptive_full(handle, cam, w, h, spp, depth, seed):
    """an adaptive frame with min_samples == samples_number: the uniform frame"""
    api.render_start_adaptive(handle, cam, api.render_params(w, h, spp, depth, seed), spp, 0.0)
    out = np.zeros((h, w, 3))
    api.render_wait(handle, out)
    return out


def _group_frame(sc, cam, w, h, spp, depth, seed):
    """trace_pixel_samples_group over the frame's own camera rays"""
    rays = _primary_rays(cam, w, h, spp, seed)
    offsets = np.arange(0, w * h * spp + 1, spp, dtype=np.uint64)
    return sc.trace_pixel_samples_group(rays, offsets, np.arange(w * h, dtype=np.uint32), depth, seed=seed).reshape(h, w, 3)


def _owner(w, h, tw, th, shards):
    """the shard that owns each pixel (rt_render_params: tile k of row ty sits at column (k % tiles_x + ty) % tiles_x)"""
    tiles_x, tiles_y = -(-w // tw), -(-h // th)
    own = np.empty((h, w), np.int64)
    for k in range(tiles_x * tiles_y):
        ty = k // tiles_x
        tx = (k % tiles_x + ty % tiles_x) % tiles_x
        own[ty * th:(ty + 1) * th, tx * tw:(tx + 1) * tw] = k % shards
    return own


def _device_accum(torch, handle, n):
    """a copy of the shard's tile-packed accumulator (n x 4 doubles), so that the next frame may reuse the handle"""
    ptr, m = api.render_device_result(handle)
    assert m == n
    if n == 0:
        return None
    return torch.as_tensor(api.DevicePointer(ptr, (n, 4)), device="cuda").clone()


# ---- scenes ------------------------------------------------------------------------------------------------------

# the camera inside an inverse_normal Lambertian sphere (albedo 0.9) with a small light: most paths bounce until the
# depth cap
CAVE = {
    "camera": {"position": [0, 0, 0], "direction": [0.3, 0.2, 1.0], "up": [0, 1, 0], "fov": 60.0, "focal_length": 1.0},
    "background": [0, 0, 0],
    "materials": {"Wall": {"type": "Lambertian", "albedo": {"type": "SolidColor", "color": [0.9, 0.9, 0.9]}},
                  "Light": {"type": "DiffuseLight", "emit": {"type": "SolidColor", "color": [4, 4, 4]}}},
    "shapes": [
        {"type": "Sphere", "name": "cave", "material": "Wall", "inverse_normal": True,
         "transform": {"translate": [0, 0, 0], "rotate": [0, 0, 0], "scale": [5, 5, 5]}},
        {"type": "Sphere", "name": "lamp", "material": "Light",
         "transform": {"translate": [1, 2, 3], "rotate": [0, 0, 0], "scale": [0.4, 0.4, 0.4]}},
    ],
}


def marched_scene(n_marched):
    """n_marched small ray-marched shapes of all six surface kinds (step 0.02, depth 2) on a grid, analytic shapes
    between them and a ground sphere"""
    kinds = list(SURFACES)
    mats = {"A": {"type": "Lambertian", "albedo": {"type": "SolidColor", "color": [0.7, 0.5, 0.3]}},
            "M": {"type": "Metal", "albedo": {"type": "SolidColor", "color": [0.8, 0.8, 0.9]}, "fuzz": 0.2},
            "G": {"type": "Dielectric", "index_of_refraction": 1.5},
            "L": {"type": "DiffuseLight", "emit": {"type": "SolidColor", "color": [3, 3, 3]}}}
    shapes = []
    for i in range(n_marched):
        r, c = divmod(i, 8)
        sc = 0.12 if kinds[i % 6] == "HuntsSurface" else 0.25
        shapes.append({"type": "BruteForsableShape", "shape": SURFACES[kinds[i % 6]], "step": 0.02, "depth": 2,
                       "material": "AMGA"[i % 4],
                       "transform": {"translate": [1.3 * c - 4.55, 1.3 * r - 2.0, 0.0], "rotate": [10.0 * i, 7.0 * i, 0],
                                     "scale": [sc, sc, sc]}})
    shapes += [
        {"type": "Sphere", "name": "s", "material": "L", "transform": {"translate": [0, 4, 1], "rotate": [0, 0, 0], "scale": [0.8] * 3}},
        {"type": "Cube", "name": "c", "material": "A", "transform": {"translate": [3, 3.5, -1], "rotate": [20, 30, 0], "scale": [0.4] * 3}},
        {"type": "Rectangle", "x0": -6, "y0": -4, "x1": 6, "y1": 5, "material": "A",
         "transform": {"translate": [0, 0, 2.0], "rotate": [0, 0, 0], "scale": [1, 1, 1]}},
        {"type": "Sphere", "name": "ground", "material": "A",
         "transform": {"translate": [0, -1003.5, 0], "rotate": [0, 0, 0], "scale": [1000] * 3}},
    ]
    return {"camera": {"position": [0.0, 0.5, -12.0], "direction": [0.0, -0.02, 1.0], "up": [0, 1, 0], "fov": 45.0,
                       "focal_length": 1.0},
            "background": [0, 0, 0], "materials": mats, "shapes": shapes}


MARCH_SCENES = {"march32": 32, "march33": 33}


# ---- depth -------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("depth", [0, 1, 2, 62])
def test_depth_edges_match_the_oracle(monkeypatch, depth):
    """max_depth 0, 1, 2 and the limit 62: the wavefront frame, the fused fallback, trace groups over the camera rays
    and the adaptive frame with min_samples == samples_number are the same frame, and it meets the strict bound"""
    w, h, spp, seed = 24, 16, 2, 77
    sc = _load("light_source.json")
    cam = sc.camera()
    frame = _frame(sc, cam, w, h, spp, depth, seed)
    check_frame(frame, po.OracleScene(sc.desc()), cam, w, h, spp, depth, seed, f"depth {depth}")
    assert np.array_equal(_group_frame(sc, cam, w, h, spp, depth, seed), frame)
    assert np.array_equal(_adaptive_full(sc.device_scene(0), cam, w, h, spp, depth, seed), frame)
    monkeypatch.setenv("RT_B200_FUSED_BOUNCE", "1")
    fused = _load("light_source.json")
    assert np.array_equal(_frame(fused, cam, w, h, spp, depth, seed), frame)


def test_depth_zero_is_the_sky_of_the_primary_ray():
    """depth 0 on an empty scene: every sample is Scene::background of its primary ray.  numpy replays ray generation
    (Philox jitter of event 0) and the sky lerp at every pixel of a 61x47 image"""
    w, h, spp, seed = 61, 47, 2, (1 << 63) + 12345
    sc = rt.Scene.from_file(scene_path("empty.json"), add_random_spheres=False)
    cam = sc.camera()
    got = _frame(sc, cam, w, h, spp, 0, seed)
    cols = np.empty((w * h, spp, 3))
    for y in range(h):
        for x in range(w):
            for s in range(spp):
                u, v = po.philox_stream(seed, x + y * w, s, 0, 2)
                d = po.get_ray(cam, w, h, x + u, y + v)[3:]
                t = 0.5 * (d[1] + 1.0)
                cols[x + y * w, s] = (1.0 - t) * np.ones(3) + t * np.array([0.5, 0.7, 1.0])
    assert check_pixels(got, cols, "depth 0 sky") == 0


def test_depth_cap_is_reached():
    """depth 62 where paths really get there: segments traced equal the oracle's, and most paths use every level"""
    w, h, spp, depth, seed = 12, 8, 2, 62, 5
    sc = rt.Scene.from_json(json.dumps(CAVE), add_random_spheres=False)
    cam = sc.camera()
    osc = po.OracleScene(sc.desc())
    sc.set_counters(True)
    sc.reset_stats()
    frame = _frame(sc, cam, w, h, spp, depth, seed)
    st = sc.stats()
    _, info = osc.render(cam, w, h, spp, depth, seed=seed, rng="philox", counters=True)
    assert st.segments == info["counters"]["segments"]
    assert st.segments > 0.5 * w * h * spp * (depth + 1), st.segments
    check_frame(frame, osc, cam, w, h, spp, depth, seed, "cave depth 62")
    assert frame.max() > 0


@pytest.mark.parametrize("depth", [0, 1, 62])
def test_segment_counts_at_depth_edges(depth):
    """the instrumented kernels trace the oracle's segments at the depth edges (depth 8: test_work_counters_match_oracle)"""
    w, h, spp, seed = 32, 24, 2, 8
    sc = _load("spheres.json")
    cam = sc.camera()
    sc.set_counters(True)
    sc.reset_stats()
    _frame(sc, cam, w, h, spp, depth, seed)
    st = sc.stats()
    _, info = po.OracleScene(sc.desc()).render(cam, w, h, spp, depth, seed=seed, rng="philox", counters=True)
    assert st.paths == w * h * spp
    assert st.segments == info["counters"]["segments"]
    assert st.segments >= w * h * spp

@pytest.mark.parametrize("bad", [63, 0xFFFFFFFE, 0xFFFFFFFF])
def test_too_deep_is_rejected(bad):
    sc = _load("spheres.json")
    cam = sc.camera()
    hd = sc.device_scene(0)
    p = api.render_params(8, 8, 2, bad, 1)
    assert _core().rt_render_start(hd, C.byref(cam), C.byref(p)) == _ffi.RT_ERR_INVALID
    ap = _ffi.AdaptiveParams(2, 0.0, 0.0)
    assert _core().rt_render_start_adaptive(hd, C.byref(cam), C.byref(p), C.byref(ap)) == _ffi.RT_ERR_INVALID
    rays = np.ascontiguousarray(_primary_rays(cam, 2, 1, 2, 1))
    offs = np.array([0, 2, 4], np.uint64)
    pix = np.array([0, 1], np.uint32)
    means = np.empty((2, 3))
    vp = lambda a: a.ctypes.data_as(C.c_void_p)
    assert _core().rt_trace_pixel_samples_group(hd, vp(rays), 4, vp(offs), vp(pix), 2, bad, 1, vp(means)) == _ffi.RT_ERR_INVALID
    # the handle is unharmed
    assert np.array_equal(_frame(sc, cam, 8, 8, 2, 62, 1), _frame(_load("spheres.json"), cam, 8, 8, 2, 62, 1))


# ---- seeds -------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", ["spheres.json", "light_source.json"])
@pytest.mark.parametrize("seed", SEEDS)
def test_seeds_across_the_64_bit_range(name, seed):
    """both words of the RNG key: per-path parity, and the frame equals the trace groups over its camera rays and the
    adaptive frame with min_samples == samples_number"""
    w, h, spp, depth = 20, 14, 2, 6
    sc = _load(name)
    cam = sc.camera()
    frame = _frame(sc, cam, w, h, spp, depth, seed)
    check_frame(frame, po.OracleScene(sc.desc()), cam, w, h, spp, depth, seed, f"{name} seed {seed}")
    assert np.array_equal(_group_frame(sc, cam, w, h, spp, depth, seed), frame)
    assert np.array_equal(_adaptive_full(sc.device_scene(0), cam, w, h, spp, depth, seed), frame)


# ---- image shapes, tiles and shards ------------------------------------------------------------------------------

@pytest.mark.parametrize("w,h", [(1, 1), (1, 45), (45, 1), (33, 31), (257, 3)])
def test_image_shapes(w, h):
    spp, depth, seed = 2, 4, 2 ** 32
    sc = _load("spheres.json")
    cam = sc.camera()
    frame = _frame(sc, cam, w, h, spp, depth, seed)
    check_frame(frame, po.OracleScene(sc.desc()), cam, w, h, spp, depth, seed, f"{w}x{h}")
    hd = sc.device_scene(0)
    for shards, tile in ((3, (7, 5)), (2, (0, 0))):
        buf = np.full((h, w, 3), -1.0)
        for s in range(shards):
            _poll_frame(hd, cam, _params(w, h, spp, depth, seed, shards, s, tile), buf)
        assert np.array_equal(buf, frame), (shards, tile)


def test_tall_image():
    """2 x 70000 (taller than a grid's 65535 rows): host poll, sharded host scatter, rt_assemble_frame and the
    multi-device handle agree bit for bit; a seeded sample of rows meets the oracle"""
    torch = pytest.importorskip("torch")
    w, h, spp, depth, seed = 2, 70000, 1, 1, 3
    sc = _load("spheres.json")
    cam = sc.camera()
    hd = sc.device_scene(0)
    frame = np.full((h, w, 3), -1.0)
    _poll_frame(hd, cam, _params(w, h, spp, depth, seed), frame)
    shards = 3
    buf = np.full((h, w, 3), -1.0)
    accs = []
    for s in range(shards):
        p = _params(w, h, spp, depth, seed, shards, s)
        _poll_frame(hd, cam, p, buf)
        accs.append(_device_accum(torch, hd, api.shard_float4_count(p, s)))
    assert np.array_equal(buf, frame)
    out = torch.full((h, w, 3), -1.0, dtype=torch.float64, device="cuda")
    api.assemble_frame(hd, _params(w, h, spp, depth, seed, shards, 0), [a.data_ptr() for a in accs], out.data_ptr())
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy(), frame)
    if rt.device_count() > 1:
        multi = rt.GpuRenderer(sc, 12, depth, seed=seed, devices=list(range(rt.device_count())))
        assert np.array_equal(multi.render(cam, w, h, spp), frame)
    rows = np.sort(np.random.default_rng(8).choice(h, 96, replace=False))
    pix = (rows[:, None] * w + np.arange(w)[None, :]).reshape(-1)
    cols = po.OracleScene(sc.desc()).frame_sample_colors(cam, w, h, spp, depth, seed, pixels=pix)
    check_pixels(frame.reshape(-1, 3)[pix], cols, "2x70000 rows")


@pytest.mark.parametrize("tile", [(1, 1), (7, 5), (31, 33), (64, 16), (40, 30)])
def test_tiles_and_shard_counts(tile):
    """every shard count 1..16 (more shards than tiles included: such a shard owns 0 slots, completes, and assembly
    never reads its buffer): the host scatter, rt_assemble_frame and the unsharded frame agree bit for bit"""
    torch = pytest.importorskip("torch")
    w, h, spp, depth, seed = 37, 23, 1, 2, 12
    sc = _load("spheres.json")
    cam = sc.camera()
    hd = sc.device_scene(0)
    ref = _frame(sc, cam, w, h, spp, depth, seed)
    tw, th = tile
    n_tiles = -(-w // tw) * -(-h // th)
    sentinel = torch.full((tw * th, 4), float("nan"), dtype=torch.float64, device="cuda")
    for shards in range(1, 17):
        buf = np.full((h, w, 3), -1.0)
        accs, total = [], 0
        for s in range(shards):
            p = _params(w, h, spp, depth, seed, shards, s, tile)
            n = api.shard_float4_count(p, s)
            total += n
            assert _poll_frame(hd, cam, p, buf) >= 0
            acc = _device_accum(torch, hd, n)
            if shards > 1 and s >= n_tiles:
                assert n == 0 and acc is None
            accs.append(acc if acc is not None else sentinel)
        assert np.array_equal(buf, ref), shards
        assert total == (w * h if shards == 1 else n_tiles * tw * th)
        out = torch.full((h, w, 3), -1.0, dtype=torch.float64, device="cuda")
        api.assemble_frame(hd, _params(w, h, spp, depth, seed, shards, 0, tile), [a.data_ptr() for a in accs],
                           out.data_ptr())
        torch.cuda.synchronize()
        assert np.array_equal(out.cpu().numpy(), ref), shards


def test_tiles_past_32_bits_are_rejected():
    sc = _load("spheres.json")
    cam = sc.camera()
    hd = sc.device_scene(0)
    for tile in ((65536, 65537), (65536, 65536), (0xFFFFFFFF, 0xFFFFFFFF)):
        p = _params(100, 100, 1, 2, 1, 2, 0, tile)
        assert _core().rt_render_start(hd, C.byref(cam), C.byref(p)) == _ffi.RT_ERR_INVALID
        assert api.shard_float4_count(p, 0) == 0
        ptrs = (C.c_void_p * 2)(8, 8)   # never dereferenced: the call fails before any launch
        assert _core().rt_assemble_frame(hd, C.byref(p), ptrs, C.c_void_p(8), None) == _ffi.RT_ERR_INVALID
    # the handle is unharmed
    assert np.array_equal(_frame(sc, cam, 9, 7, 1, 2, 1), _frame(_load("spheres.json"), cam, 9, 7, 1, 2, 1))


# ---- batching ----------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("batch", [1, 7, 1000])
@pytest.mark.parametrize("lanes", [1, 2, 4])
def test_batch_splits(monkeypatch, batch, lanes):
    """RT_B200_BATCH_PATHS with spp 3 (batches of whole pixels that split tile rows), 1, 2 or 4 lanes; delivered through
    a render_poll loop into a buffer of -1: the default frame bit for bit, unsharded and sharded, and the pixels of
    other shards stay -1"""
    w, h, spp, depth, seed = 23, 13, 3, 2, 4
    ref_sc = _load("spheres.json")
    cam = ref_sc.camera()
    ref = _frame(ref_sc, cam, w, h, spp, depth, seed)
    monkeypatch.setenv("RT_B200_LANES", str(lanes))
    monkeypatch.setenv("RT_B200_BATCH_PATHS", str(batch))
    sc = _load("spheres.json")
    hd = sc.device_scene(0)
    buf = np.full((h, w, 3), -1.0)
    _poll_frame(hd, cam, _params(w, h, spp, depth, seed), buf)
    assert np.array_equal(buf, ref)
    shards, tile = 3, (7, 5)
    own = _owner(w, h, *tile, shards)
    for s in range(shards):
        buf = np.full((h, w, 3), -1.0)
        _poll_frame(hd, cam, _params(w, h, spp, depth, seed, shards, s, tile), buf)
        assert np.array_equal(buf[own == s], ref[own == s]), s
        assert (buf[own != s] == -1.0).all(), s


def test_accumulation_with_changing_sample_counts():
    """frames of 1, 3 and 2 samples accumulate to the 6-sample frame bit for bit, unsharded and as 3 shards of 7x5
    tiles, and meet the strict bound against the oracle's samples 0..5"""
    w, h, depth, seed = 23, 13, 4, (1 << 63) + 12345
    sc = _load("spheres.json")
    cam = sc.camera()
    ref6 = _frame(sc, cam, w, h, 6, depth, seed)
    check_frame(ref6, po.OracleScene(sc.desc()), cam, w, h, 6, depth, seed, "accumulated 1+3+2")
    for shards, tile in ((1, (0, 0)), (3, (7, 5))):
        buf = np.full((h, w, 3), -1.0)
        for s in range(shards):
            shard_sc = _load("spheres.json")
            hd = shard_sc.device_scene(0)
            api.render_set_accumulate(hd, True)
            for spp in (1, 3, 2):
                _poll_frame(hd, cam, _params(w, h, spp, depth, seed, shards, s, tile), buf)
            assert api.render_accumulated_samples(hd) == 6
        assert np.array_equal(buf, ref6), shards


# ---- the 32 / 33 marched-shape boundary --------------------------------------------------------------------------

@pytest.mark.parametrize("name", ["march32", "march33"])
def test_marched_shape_boundary(name):
    """bit 31 of the march mask (32 marched shapes) and the fused fallback a 33rd selects: nearest hit bit for bit,
    VERIFY clean, frames under the strict bound, trace groups equal to the frame; the fallback cannot accumulate or
    render adaptively"""
    sc = _load(name)
    assert int((sc.shape_kinds() == _ffi.RT_SHAPE_MARCH).sum()) == MARCH_SCENES[name]
    cam = sc.camera()
    osc = po.OracleScene(sc.desc())
    rays = scene_rays(sc, 2000, seed=4)
    want = osc.intersect_batch(rays)
    assert set(range(MARCH_SCENES[name])) <= set(want["index"].tolist())   # every marched shape, bit 31 included
    for mode in (rt.RT_ISECT_BRUTE, rt.RT_ISECT_FAST):
        _compare(sc.closest_hit(rays, mode=mode), want, len(rays), mode)
    sc.reset_stats()
    sc.closest_hit(rays, mode=rt.RT_ISECT_VERIFY, want=("index",))
    st = sc.stats()
    assert st.verify_rays == 0 and st.verify_false_culls == 0
    w, h, spp, depth, seed = 24, 18, 2, 2, 9
    frame = _frame(sc, cam, w, h, spp, depth, seed)
    check_frame(frame, osc, cam, w, h, spp, depth, seed, name)
    assert np.array_equal(_group_frame(sc, cam, w, h, spp, depth, seed), frame)
    hd = sc.device_scene(0)
    if name == "march33":
        assert _core().rt_render_set_accumulate(hd, 1) == _ffi.RT_ERR_STATE
        p = api.render_params(w, h, spp, depth, seed)
        ap = _ffi.AdaptiveParams(2, 0.0, 0.0)
        assert _core().rt_render_start_adaptive(hd, C.byref(cam), C.byref(p), C.byref(ap)) == _ffi.RT_ERR_STATE
    else:
        assert np.array_equal(_adaptive_full(hd, cam, w, h, spp, depth, seed), frame)


# ---- device entry points -----------------------------------------------------------------------------------------

def test_intersect_batch_device_streams_and_null_outputs():
    """rt_intersect_batch_device on the library's stream (NULL), the legacy default stream (0x1) and a torch side
    stream, with some outputs NULL: the host form bit for bit"""
    torch = pytest.importorskip("torch")
    sc = _load("cornell_box.json")
    rays = scene_rays(sc, 4096, seed=2)
    want = sc.closest_hit(rays, mode=rt.RT_ISECT_FAST)
    d_rays = torch.from_numpy(rays).cuda()
    n = len(rays)
    side = torch.cuda.Stream()
    hd = sc.device_scene(0)
    for stream in (None, 1, side.cuda_stream):
        for keys in (("index", "t", "normal", "point", "uv", "front"), ("index", "t"), ("normal", "uv"), ("front",)):
            out = {"index": torch.full((n,), -7, dtype=torch.int32, device="cuda"),
                   "t": torch.zeros(n, dtype=torch.float64, device="cuda"),
                   "normal": torch.zeros((n, 3), dtype=torch.float64, device="cuda"),
                   "point": torch.zeros((n, 3), dtype=torch.float64, device="cuda"),
                   "uv": torch.zeros((n, 2), dtype=torch.float64, device="cuda"),
                   "front": torch.zeros(n, dtype=torch.uint8, device="cuda")}
            torch.cuda.synchronize()
            ptr = lambda k: out[k].data_ptr() if k in keys else None
            rc = _core().rt_intersect_batch_device(hd, d_rays.data_ptr(), n, 0.001, float("inf"), rt.RT_ISECT_FAST,
                                                   ptr("index"), ptr("t"), ptr("normal"), ptr("point"), ptr("uv"),
                                                   ptr("front"), stream)
            assert rc == 0
            torch.cuda.synchronize()
            hit = want["index"] >= 0
            for k in keys:
                g = out[k].cpu().numpy()
                if k in ("index",):
                    assert np.array_equal(g, want[k]), (stream, k)
                else:
                    assert np.array_equal(g[hit], want[k][hit], equal_nan=True), (stream, k)


def test_device_frame_is_the_polled_frame():
    torch = pytest.importorskip("torch")
    w, h, spp, depth, seed = 40, 30, 2, 6, 1 << 32
    sc = _load("cornell_box.json")
    cam = sc.camera()
    hd = sc.device_scene(0)
    buf = np.full((h, w, 3), -1.0)
    _poll_frame(hd, cam, _params(w, h, spp, depth, seed), buf)
    ptr, n = C.c_void_p(), C.c_uint64()
    assert _core().rt_render_device_frame(hd, C.byref(ptr), C.byref(n)) == 0
    assert n.value == w * h
    d = torch.as_tensor(api.DevicePointer(ptr.value, (n.value, 3)), device="cuda").cpu().numpy()
    assert np.array_equal(d.reshape(h, w, 3), buf)
