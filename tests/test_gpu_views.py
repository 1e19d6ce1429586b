"""rt_render_start_views: several cameras of one scene in one frame.

View v of a views frame must equal, bit for bit, the rt_render_start frame of cameras[v] with the same params -- whatever
the batch size, the lanes, the kernel timing, the fused fallback, the devices or the shards.  The frame is the stacked
image (w, n_views*h), view v in rows v*h .. v*h+h-1.
"""
import ctypes as C
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest

import rs_pathtracing_b200 as rt
from rs_pathtracing_b200 import _ffi, api
from oracle import pyoracle as po

from conftest import scene_path
from test_gpu_adaptive import _variant_4b
from test_gpu_frame_edges import _device_accum, _owner, _params, check_frame, marched_scene

pytestmark = pytest.mark.gpu

DEPTH = 8
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _load(name, variant=""):
    if name == "march33":
        sc = rt.Scene.from_json(json.dumps(marched_scene(33)), add_random_spheres=False)
        return sc, sc.camera()
    sc = rt.Scene.from_file(scene_path(name), random_spheres_seed=1)
    return sc, (_variant_4b(sc) if variant == "4b" else sc.camera())


def _views(hd, cams, w, h, spp, depth=DEPTH, seed=5, shards=1, index=0, tile=(0, 0), fill=0.0):
    """one views frame through the raw calls, waited for into a (V, h, w, 3) buffer of `fill`"""
    api.render_start_views(hd, cams, _params(w, h, spp, depth, seed, shards, index, tile))
    out = np.full((len(cams), h, w, 3), fill)
    api.render_wait(hd, out)
    return out


def _frames(hd, cams, w, h, spp, depth=DEPTH, seed=5):
    """what the contract says: the rt_render_start frame of every camera; hd: a device handle, or a Scene (its device-0
    handle, the Scene kept alive meanwhile)"""
    if isinstance(hd, rt.Scene):
        sc, hd = hd, hd.device_scene(0)
    out = np.zeros((len(cams), h, w, 3))
    for v, cam in enumerate(cams):
        api.render_start(hd, cam, api.render_params(w, h, spp, depth, seed))
        api.render_wait(hd, out[v])
    return out


def _fresh(name, variant=""):
    """a Scene of its own, so a device handle of its own, for the reference frames (its handle lives as long as it)"""
    return _load(name, variant)[0]


def _stereo(cam):
    pos, right = np.array(cam.position.tuple()), np.array(cam.right.tuple())
    d, up = cam.direction.tuple(), cam.up.tuple()
    return [rt.camera_new(pos + s * 0.065 * right, d, up, cam.focal_length, cam.fov_rad) for s in (-0.5, 0.5)]


def _cube(cam):
    pos = cam.position.tuple()
    dirs = [((1, 0, 0), (0, 1, 0)), ((-1, 0, 0), (0, 1, 0)), ((0, 1, 0), (0, 0, -1)), ((0, -1, 0), (0, 0, 1)),
            ((0, 0, 1), (0, 1, 0)), ((0, 0, -1), (0, 1, 0))]
    return [rt.camera_new(pos, d, up, 1.0, math.pi / 2) for d, up in dirs]


def _random_orbit(cam, n, seed=3):
    """n orbit cameras in a random order, every third with another fov and every fourth with another focal length"""
    rng = np.random.default_rng(seed)
    cams = api.orbit_cameras(cam, n)
    out = []
    for k in rng.permutation(n):
        c = cams[k]
        fov = c.fov_rad * (0.6 if k % 3 == 0 else 1.0)
        focal = c.focal_length * (2.5 if k % 4 == 0 else 1.0)
        out.append(rt.camera_new(c.position.tuple(), c.direction.tuple(), c.up.tuple(), focal, fov))
    return out


CAMERA_SETS = {
    "one": lambda cam: [cam],
    "stereo": _stereo,
    "cube": _cube,
    "orbit16": lambda cam: _random_orbit(cam, 16),
    "repeated": lambda cam: [cam, cam, cam],
}


# ---- the frame ---------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name,variant", [("spheres.json", ""), ("cornell_box.json", ""), ("dupin.json", ""),
                                          ("detached_materials.json", "4b")])
@pytest.mark.parametrize("camera_set", list(CAMERA_SETS))
def test_every_view_is_its_frame(name, variant, camera_set):
    w, h, spp = 40, 30, 2
    sc, cam = _load(name, variant)
    cams = CAMERA_SETS[camera_set](cam)
    got = _views(sc.device_scene(0), cams, w, h, spp)
    assert np.array_equal(got, _frames(_fresh(name, variant), cams, w, h, spp))


def test_views_against_the_oracle():
    """four orbit views, each within one float ulp per path of the oracle's samples of its own camera"""
    w, h, spp, seed = 24, 18, 3, 11
    sc, cam = _load("spheres.json")
    cams = api.orbit_cameras(cam, 4)
    got = _views(sc.device_scene(0), cams, w, h, spp, seed=seed)
    osc = po.OracleScene(sc.desc())
    for v, c in enumerate(cams):
        check_frame(got[v], osc, c, w, h, spp, DEPTH, seed, f"view {v}")


def test_renderer_views():
    w, h, spp, seed = 48, 32, 2, 4
    sc, cam = _load("cornell_box.json")
    cams = _random_orbit(cam, 5)
    ren = rt.GpuRenderer(sc, 12, DEPTH, seed=seed)
    got = ren.render_views(cams, w, h, spp)
    assert got.shape == (5, h, w, 3)
    ref_sc, _ = _load("cornell_box.json")
    ref = rt.GpuRenderer(ref_sc, 12, DEPTH, seed=seed)
    for v, c in enumerate(cams):
        assert np.array_equal(got[v], ref.render(c, w, h, spp)), v


# ---- schedules ---------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", ["spheres.json", "march33"])
def test_schedules_give_the_same_frame(monkeypatch, name):
    """batches of 1 and 7 paths, one view's paths - 1, + 1 and a batch of 1.5 views (batches across view boundaries),
    1 / 2 / 3 lanes, kernel timing on, the fused k_bounce: the same views, bit for bit, also when polled"""
    w, h, spp, seed = 16, 12, 2, 21
    sc, cam = _load(name)
    cams = _random_orbit(cam, 3, seed=8)
    ref = _frames(sc.device_scene(0), cams, w, h, spp, seed=seed)
    view_paths = w * h * spp

    def run(env, timing=False):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        alt, _ = _load(name)   # a new device handle reads the variables
        hd = alt.device_scene(0)
        if timing:
            alt.set_kernel_timing(True, 0)
        api.render_start_views(hd, cams, api.render_params(w, h, spp, DEPTH, seed))
        buf = np.full((len(cams), h, w, 3), -1.0)
        while not api.render_poll(hd, buf):
            pass
        if timing:
            s = alt.stats(0)
            assert s.ms_raygen > 0 and s.ms_resolve > 0 and s.launches_extend > 0
        for k in env:
            monkeypatch.delenv(k)
        return buf

    assert np.array_equal(run({}), ref)
    for env in ({"RT_B200_BATCH_PATHS": "1"}, {"RT_B200_BATCH_PATHS": "7"},
                {"RT_B200_BATCH_PATHS": str(view_paths - 1)}, {"RT_B200_BATCH_PATHS": str(view_paths + 1)},
                {"RT_B200_BATCH_PATHS": str(view_paths * 3 // 2)},
                {"RT_B200_BATCH_PATHS": "100", "RT_B200_LANES": "1"},
                {"RT_B200_BATCH_PATHS": "100", "RT_B200_LANES": "2"}, {"RT_B200_BATCH_PATHS": "100", "RT_B200_LANES": "3"},
                {"RT_B200_FUSED_BOUNCE": "1"}, {"RT_B200_FUSED_BOUNCE": "1", "RT_B200_BATCH_PATHS": "7"}):
        assert np.array_equal(run(env), ref), env
    assert np.array_equal(run({"RT_B200_BATCH_PATHS": "7"}, timing=True), ref)


# ---- delivery ----------------------------------------------------------------------------------------------------

def test_delivery(monkeypatch):
    """pixels a poll delivers before done are final, in the v*w*h + x + y*w layout; the device frame covers every view;
    the device tone map equals rt_tonemap_rgba8 of the views"""
    monkeypatch.setenv("RT_B200_BATCH_PATHS", "1000")
    sc, cam = _load("cornell_box.json")
    hd = sc.device_scene(0)
    w, h, spp = 50, 40, 4
    cams = api.orbit_cameras(cam, 4)
    ref = _frames(_fresh("cornell_box.json"), cams, w, h, spp)
    api.render_start_views(hd, cams, api.render_params(w, h, spp, DEPTH, 5))
    buf = np.full(len(cams) * w * h * 3, -7.0)
    done = api.render_poll(hd, buf)
    while not done:
        view = buf.reshape(-1, 3)
        seen = ~(view == -7.0).all(axis=1)
        assert np.array_equal(view[seen], ref.reshape(-1, 3)[seen])
        done = api.render_poll(hd, buf)
    assert np.array_equal(buf.reshape(ref.shape), ref)

    ptr, n = C.c_void_p(), C.c_uint64()
    assert _ffi.core().rt_render_device_frame(hd, C.byref(ptr), C.byref(n)) == _ffi.RT_OK
    assert n.value == len(cams) * w * h
    torch = pytest.importorskip("torch")
    dev = torch.as_tensor(api.DevicePointer(ptr.value, (n.value, 3)), device="cuda").cpu().numpy()
    assert np.array_equal(dev.reshape(ref.shape), ref)
    assert np.array_equal(api.tonemap_last_frame(hd).reshape(len(cams), h, w, 4), rt.tonemap_rgba8(sc, ref))


# ---- devices and shards ------------------------------------------------------------------------------------------

@pytest.mark.parametrize("tile", [(16, 16), (32, 32)])
def test_explicit_shards_assemble_to_the_frame(tile):
    """shards 2, 4, 8 and 16 of the stacked image (h not a multiple of the tile: tiles straddle two views): each shard's
    polled pixels, and rt_assemble_frame over the gathered accumulators with the stacked params, are the unsharded views
    frame bit for bit"""
    torch = pytest.importorskip("torch")
    w, h, spp, seed = 37, 23, 2, 12
    sc, cam = _load("spheres.json")
    hd = sc.device_scene(0)
    cams = _random_orbit(cam, 3, seed=5)
    ref = _views(hd, cams, w, h, spp, seed=seed).reshape(-1, w, 3)
    V, H = len(cams), len(cams) * h
    tw, th = tile
    sentinel = torch.full((tw * th, 4), float("nan"), dtype=torch.float64, device="cuda")
    sc.reset_stats(0)
    for shards in (2, 4, 8, 16):
        own = _owner(w, H, tw, th, shards)
        accs = []
        for s in range(shards):
            p = _params(w, h, spp, DEPTH, seed, shards, s, tile)
            n = api.shard_float4_count(api.stacked_params(p, V), s)
            buf = np.full((H, w, 3), -1.0)
            api.render_start_views(hd, cams, p)
            while not api.render_poll(hd, buf):
                pass
            assert np.array_equal(buf[own == s], ref[own == s]), (shards, s)
            assert (buf[own != s] == -1.0).all(), (shards, s)
            acc = _device_accum(torch, hd, n)
            accs.append(acc if acc is not None else sentinel)
        out = torch.full((H, w, 3), -1.0, dtype=torch.float64, device="cuda")
        api.assemble_frame(hd, api.stacked_params(_params(w, h, spp, DEPTH, seed, shards, 0, tile), V),
                           [a.data_ptr() for a in accs], out.data_ptr())
        torch.cuda.synchronize()
        assert np.array_equal(out.cpu().numpy(), ref), shards
    # every shard counts its real pixels only: each set of shards adds the frame's paths once
    assert sc.stats(0).paths == 4 * V * w * h * spp


def test_multi_device_handle():
    n = rt.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    w, h, spp, seed = 120, 70, 2, 8
    sc, cam = _load("cornell_box.json")
    cams = _random_orbit(cam, 6)
    ref = _views(sc.device_scene(0), cams, w, h, spp, seed=seed)
    hm = sc.device_scene_multi(list(range(n)))
    assert np.array_equal(_views(hm, cams, w, h, spp, seed=seed), ref)
    ren = rt.GpuRenderer(sc, 12, DEPTH, seed=seed, devices=list(range(n)))
    assert np.array_equal(ren.render_views(cams, w, h, spp), ref)


def test_distributed_renderer_views():
    """DistributedRenderer.render_views under torchrun over every GPU of the box (one rank when there is one)"""
    torch = pytest.importorskip("torch")
    tool = os.path.join(ROOT, "tools", "check_distributed_views.py")
    n = max(1, min(torch.cuda.device_count(), 8))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr",
           "127.0.0.1", "--master-port", "29562", tool]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert r.stdout.count("identical") == 3, r.stdout[-3000:]


# ---- edges -------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("w,h,n_views", [(1, 1, 5), (4, 4, 4096)])
def test_view_shapes(w, h, n_views):
    sc, cam = _load("spheres.json")
    cams = _random_orbit(cam, n_views, seed=n_views)
    got = _views(sc.device_scene(0), cams, w, h, 2, depth=4)
    # (the 4096-view frame is checked on a sample of its views)
    pick = range(n_views) if n_views <= 8 else sorted({0, 1, 777, 2048, n_views - 2, n_views - 1})
    ref = _frames(_fresh("spheres.json"), [cams[v] for v in pick], w, h, 2, depth=4)
    assert np.array_equal(got[list(pick)], ref)


@pytest.mark.parametrize("depth", [0, 1, 62])
def test_depths(depth):
    sc, cam = _load("cornell_box.json")
    cams = _random_orbit(cam, 3)
    assert np.array_equal(_views(sc.device_scene(0), cams, 32, 24, 2, depth=depth),
                          _frames(_fresh("cornell_box.json"), cams, 32, 24, 2, depth=depth))


@pytest.mark.parametrize("seed", [0, (1 << 64) - 1])
@pytest.mark.parametrize("spp", [1, 3])
def test_seeds_and_one_sample(seed, spp):
    sc, cam = _load("spheres.json")
    cams = _stereo(cam)
    assert np.array_equal(_views(sc.device_scene(0), cams, 32, 24, spp, seed=seed),
                          _frames(_fresh("spheres.json"), cams, 32, 24, spp, seed=seed))


def test_size_limits():
    """n_views*h and n_views*w*h at their limits: one above is RT_ERR_INVALID and leaves the last frame alone; one below
    is accepted (rendered here as a shard that owns no tile)"""
    sc, cam = _load("spheres.json")
    hd = sc.device_scene(0)
    lib = _ffi.core()
    small = _views(hd, [cam, cam], 8, 6, 1)
    m = 2**32 - 1   # = 3 * 5 * 17 * 257 * 65537

    def start(n_views, w, h, shards=1, index=0, tile=(0, 0)):
        cams = (_ffi.Camera * n_views)(*([cam] * n_views))
        return lib.rt_render_start_views(hd, cams, n_views, C.byref(_params(w, h, 1, 0, 0, shards, index, tile)))

    def last_frame_pixels():
        ptr, n = C.c_void_p(), C.c_uint64()
        assert lib.rt_render_device_frame(hd, C.byref(ptr), C.byref(n)) == _ffi.RT_OK
        return n.value

    assert start(3, 1, m // 3 + 1) == _ffi.RT_ERR_INVALID            # n_views*h = 2^32 + 2
    assert start(2, 1, 2**31) == _ffi.RT_ERR_INVALID                 # n_views*h = 2^32
    assert start(3, 5, m // 15 + 1) == _ffi.RT_ERR_INVALID           # n_views*w*h = 2^32 + 14
    assert start(4, 2**16, 2**14) == _ffi.RT_ERR_INVALID             # n_views*w*h = 2^32
    assert last_frame_pixels() == 2 * 8 * 6
    assert np.array_equal(api.tonemap_last_frame(hd).reshape(2, 6, 8, 4), rt.tonemap_rgba8(sc, small))
    # one below: 16 shards of tiles of 2^31 (2^29) rows -- the stacked image has 2 tiles, shard 5 owns none
    for n_views, w, h, tile in ((3, 1, m // 3, (1, 2**31)), (3, 5, m // 15, (5, 2**29))):
        assert start(n_views, w, h, 16, 5, tile) == _ffi.RT_OK, (n_views, w, h)
        assert lib.rt_render_wait(hd, None) == _ffi.RT_OK
        ptr, n = api.render_device_result(hd)
        assert n == 0


# ---- state -------------------------------------------------------------------------------------------------------

def test_state(monkeypatch):
    """a new start stops a frame in flight; stop drains the frame; paths; pixel stats refuse; caller rays refuse while
    the frame is in flight; an accumulating frame after a views frame starts afresh"""
    monkeypatch.setenv("RT_B200_BATCH_PATHS", "2000")
    sc, cam = _load("cornell_box.json")
    hd = sc.device_scene(0)
    w, h, spp = 60, 40, 4
    cams = api.orbit_cameras(cam, 3)
    ref = _frames(_fresh("cornell_box.json"), cams, w, h, spp)
    lib = _ffi.core()

    sc.reset_stats(0)
    api.render_start_views(hd, cams, api.render_params(w, h, spp, DEPTH, 5))
    rays = api.make_rays(np.array([cam.position.tuple()]), np.array([cam.direction.tuple()]))
    off, pix, means = np.array([0, 1], np.uint64), np.zeros(1, np.uint32), np.empty((1, 3))
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    assert lib.rt_trace_pixel_samples_group(hd, p(rays), 1, p(off), p(pix), 1, DEPTH, 0, p(means)) == _ffi.RT_ERR_STATE
    out = np.zeros_like(ref)
    api.render_wait(hd, out)
    assert np.array_equal(out, ref)
    assert sc.stats(0).paths == len(cams) * w * h * spp
    assert lib.rt_render_pixel_stats(hd, p(np.empty(len(cams) * w * h, np.uint32)), None) == _ffi.RT_ERR_STATE

    # a start while a frame is in flight stops it first; so does a views start after a frame
    api.render_start(hd, cam, api.render_params(w, h, 64, DEPTH, 5))
    assert np.array_equal(_views(hd, cams, w, h, spp), ref)
    api.render_start_views(hd, cams, api.render_params(w, h, 64, DEPTH, 5))
    api.render_start_views(hd, cams, api.render_params(w, h, spp, DEPTH, 5))
    out[:] = 0
    api.render_wait(hd, out)
    assert np.array_equal(out, ref)

    api.render_start_views(hd, cams, api.render_params(w, h, spp, DEPTH, 5))
    assert lib.rt_render_stop(hd) == _ffi.RT_OK
    with pytest.raises(rt.RtError):
        api.render_poll(hd, out)

    api.render_set_accumulate(hd, True)
    a = _frames(hd, [cams[0]], w, h, 4)
    assert api.render_accumulated_samples(hd) == 4
    _views(hd, cams, w, h, spp)
    assert api.render_accumulated_samples(hd) == 0
    assert np.array_equal(_frames(hd, [cams[0]], w, h, 4), a)
    assert api.render_accumulated_samples(hd) == 4
    api.render_set_accumulate(hd, False)
    # a frame after a views frame keeps its pixel statistics again
    counts, _ = api.render_pixel_stats(hd)
    assert (counts == 4).all()


def test_bad_input_is_rejected():
    sc, cam = _load("spheres.json")
    hd = sc.device_scene(0)
    w, h = 8, 6
    cams = (_ffi.Camera * 2)(cam, cam)
    lib = _ffi.core()

    def start(p, c=cams, n=2):
        return lib.rt_render_start_views(hd, c, n, C.byref(p))

    assert start(api.render_params(w, h, 4, DEPTH), None) == _ffi.RT_ERR_INVALID        # NULL cameras
    assert start(api.render_params(w, h, 4, DEPTH), n=0) == _ffi.RT_ERR_INVALID         # no views
    assert start(api.render_params(w, h, 0, DEPTH)) == _ffi.RT_ERR_INVALID              # 0 samples
    assert start(api.render_params(0, h, 4, DEPTH)) == _ffi.RT_ERR_INVALID              # empty view
    assert start(api.render_params(w, 0, 4, DEPTH)) == _ffi.RT_ERR_INVALID
    assert start(api.render_params(w, h, 4, 63)) == _ffi.RT_ERR_INVALID                 # depth 63
    assert start(api.render_params(w, h, 4, DEPTH, 0, 4, 4)) == _ffi.RT_ERR_INVALID     # shard_index >= shard_count
    assert start(api.render_params(w, h, 4, DEPTH, 0, 17, 0)) == _ffi.RT_ERR_INVALID    # more than 16 shards
    for bad in ([], [cam, None], cam):
        with pytest.raises(ValueError):
            api.render_start_views(hd, bad, api.render_params(w, h, 4, DEPTH))
    # the handle is unharmed
    assert np.array_equal(_views(hd, [cam, cam], w, h, 4), _frames(hd, [cam, cam], w, h, 4))
