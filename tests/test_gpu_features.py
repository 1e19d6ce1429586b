"""rt_render_start_features: the rt_render_start frame with per-pixel features of the first hit of each sample's camera ray.

The frame of a features frame must be rt_render_start's bit for bit, and every feature must equal, bit for bit,
api.feature_means over the frame's own camera rays (api.primary_rays) -> Scene.closest_hit (index, t, normal) and
Scene.scatter(level=0) (color) -- whatever the depth, the batch size, the lanes, the kernel timing, the fused fallback,
the devices or the shards.  The nearest hits are in turn pinned to the oracle on spp-1 frames.
"""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import rs_pathtracing_b200 as rt
from rs_pathtracing_b200 import _ffi, api
from oracle import pyoracle as po

from conftest import scene_path
from test_gpu_frame_edges import _owner, _params, marched_scene
from test_gpu_render import _variant_4b
from test_gpu_scene_update import Edited, create, update_transforms

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCENES = ["spheres.json", "cornell_box.json", "dupin.json", "4b", "light_source.json", "torus.json", "march33"]


def same(a, b):
    """bit for bit, NaN payloads and signed zeros included"""
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and a.tobytes() == b.tobytes()


def same_features(a, b):
    return set(a) == set(b) == set(api.FEATURE_NAMES) and all(same(a[k], b[k]) for k in api.FEATURE_NAMES)


def _load(name):
    if name == "march33":   # 33 ray-marched shapes: the fused k_bounce renders it
        sc = rt.Scene.from_json(json.dumps(marched_scene(33)), add_random_spheres=False)
        return sc, sc.camera()
    if name == "4b":
        sc = rt.Scene.from_file(scene_path("detached_materials.json"), random_spheres_seed=1)
        return sc, _variant_4b(sc)
    sc = rt.Scene.from_file(scene_path(name), random_spheres_seed=1)
    return sc, sc.camera()


def _features(hd, cam, w, h, spp, depth, seed, shards=1, index=0, tile=(0, 0)):
    """one features frame through the raw calls: (frame polled into a buffer of -1, features) -- None for a shard"""
    api.render_start_features(hd, cam, _params(w, h, spp, depth, seed, shards, index, tile))
    frame = np.full((h, w, 3), -1.0)
    while not api.render_poll(hd, frame):
        pass
    return frame, (api.render_features(hd) if shards == 1 else None)


def _plain(hd, cam, w, h, spp, depth, seed):
    api.render_start(hd, cam, api.render_params(w, h, spp, depth, seed))
    frame = np.zeros((h, w, 3))
    api.render_wait(hd, frame)
    return frame


def _replay(sc, cam, w, h, spp, seed):
    """the contract restated: the frame's own camera rays through closest_hit and scatter at level 0"""
    rays, keys = api.primary_rays(cam, w, h, np.arange(w * h), spp, seed)
    hit = sc.closest_hit(rays, mode=rt.RT_ISECT_FAST, want=("index", "t", "normal"))
    color = sc.scatter(rays, keys, 0, seed)["color"]
    m = api.feature_means(hit["index"], hit["t"], hit["normal"], color, np.arange(0, w * h * spp + 1, spp))
    return {k: v.reshape((h, w) + v.shape[1:]) for k, v in m.items()}


# ---- the contract --------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", SCENES)
def test_features_replay_the_hit_and_scatter_queries(name):
    """depths 0, 1, 8, 62 and seeds 0, 2^64-1: the frame is rt_render_start's, and the features are feature_means over
    closest_hit + scatter(level 0) of the frame's camera rays, bit for bit, the same at every depth"""
    w, h, spp = 14, 10, 3
    sc, cam = _load(name)
    hd = sc.device_scene(0)
    for seed in (0, (1 << 64) - 1):
        want = _replay(sc, cam, w, h, spp, seed)
        for depth in (0, 1, 8, 62):
            frame, feats = _features(hd, cam, w, h, spp, depth, seed)
            assert same(frame, _plain(hd, cam, w, h, spp, depth, seed)), (name, seed, depth)
            assert same_features(feats, want), (name, seed, depth)
        cov = want["coverage"]
        assert ((cov >= 0) & (cov <= 1)).all()
        assert np.isposinf(want["depth"][cov == 0]).all() and (want["shape"][cov == 0] == -1).all()


def test_device_frame_and_tone_map_are_the_plain_frames():
    sc, cam = _load("cornell_box.json")
    hd = sc.device_scene(0)
    w, h, spp, depth, seed = 24, 18, 4, 8, 5
    plain = _plain(hd, cam, w, h, spp, depth, seed)
    lib = _ffi.core()
    ptr, cnt = C.c_void_p(), C.c_uint64()
    assert lib.rt_render_device_frame(hd, C.byref(ptr), C.byref(cnt)) == _ffi.RT_OK
    tone_plain = api.tonemap_last_frame(hd, w * h)
    frame, _ = _features(hd, cam, w, h, spp, depth, seed)
    assert same(frame, plain)
    assert lib.rt_render_device_frame(hd, C.byref(ptr), C.byref(cnt)) == _ffi.RT_OK and cnt.value == w * h
    assert same(api.tonemap_last_frame(hd, w * h), tone_plain)


# ---- schedules -----------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", ["cornell_box.json", "march33"])
def test_schedules_give_the_same_features(monkeypatch, name):
    """batches of 1 and 7 paths and of one pixel's paths - 1 / + 1, 1 / 2 / 3 lanes, kernel timing and counters, the
    fused k_bounce"""
    w, h, spp, depth, seed = 16, 12, 5, 8, 21
    sc, cam = _load(name)
    ref_frame, ref = _features(sc.device_scene(0), cam, w, h, spp, depth, seed)

    def run(env, timing=False):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        alt, _ = _load(name)   # a new device handle reads the variables
        hd = alt.device_scene(0)
        if timing:
            alt.set_kernel_timing(True, 0)
            alt.set_counters(True, 0)
        out = _features(hd, cam, w, h, spp, depth, seed)
        if timing:
            s = alt.stats(0)
            assert s.ms_resolve > 0 and s.launches_extend > 0 and s.segments > 0
        for k in env:
            monkeypatch.delenv(k)
        return out

    for env in ({"RT_B200_BATCH_PATHS": "1"}, {"RT_B200_BATCH_PATHS": "7"},
                {"RT_B200_BATCH_PATHS": str(spp - 1)}, {"RT_B200_BATCH_PATHS": str(spp + 1)},
                {"RT_B200_BATCH_PATHS": "100", "RT_B200_LANES": "1"},
                {"RT_B200_BATCH_PATHS": "100", "RT_B200_LANES": "2"}, {"RT_B200_BATCH_PATHS": "100", "RT_B200_LANES": "3"},
                {"RT_B200_FUSED_BOUNCE": "1"}, {"RT_B200_FUSED_BOUNCE": "1", "RT_B200_BATCH_PATHS": "7"}):
        frame, feats = run(env)
        assert same(frame, ref_frame) and same_features(feats, ref), env
    frame, feats = run({"RT_B200_BATCH_PATHS": "7"}, timing=True)
    assert same(frame, ref_frame) and same_features(feats, ref)


@pytest.mark.parametrize("spp", [63, 64, 65])
def test_samples_near_the_batch_cap(monkeypatch, spp):
    """a batch of 64 paths: a pixel's samples fill it, overflow it by one (one pixel per batch) or leave one slot"""
    monkeypatch.setenv("RT_B200_BATCH_PATHS", "64")
    sc, cam = _load("dupin.json")
    w, h, depth, seed = 5, 3, 4, 17
    frame, feats = _features(sc.device_scene(0), cam, w, h, spp, depth, seed)
    assert same_features(feats, _replay(sc, cam, w, h, spp, seed))
    assert same(frame, _plain(sc.device_scene(0), cam, w, h, spp, depth, seed))


# ---- images --------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("w,h,spp", [(1, 1, 1), (1, 1, 9), (33, 17, 1), (33, 17, 2), (45, 1, 3), (1, 45, 3)])
def test_image_shapes(w, h, spp):
    sc, cam = _load("spheres.json")
    hd = sc.device_scene(0)
    depth, seed = 8, 9
    frame, feats = _features(hd, cam, w, h, spp, depth, seed)
    dev = api.render_features(hd, device=True)
    assert set(dev) == set(api.FEATURE_NAMES) and all(dev.values())
    assert same_features(feats, _replay(sc, cam, w, h, spp, seed))
    assert same(frame, _plain(hd, cam, w, h, spp, depth, seed))


# ---- devices and shards --------------------------------------------------------------------------------------------

def _padding(w, h, tw, th, shards, s, n_slots):
    """the owned slots of shard s that are padding of clipped border tiles (ShardMap::pixel_of)"""
    tiles_x = -(-w // tw)
    q = np.arange(n_slots)
    j, r = q // (tw * th), q % (tw * th)
    k = s + j * shards
    ty = k // tiles_x
    tx = (k % tiles_x + ty % tiles_x) % tiles_x
    return (tx * tw + r % tw >= w) | (ty * th + r // tw >= h)


@pytest.mark.parametrize("tile", [(16, 16), (7, 5)])
def test_explicit_shards_assemble_to_the_features(tile):
    """shards 2, 3, 5 (clipped border tiles): each shard's polled pixels are the frame's, padding slots hold zero sums
    and shape -1, and rt_assemble_features over the gathered sums is the unsharded features frame bit for bit"""
    torch = pytest.importorskip("torch")
    w, h, spp, depth, seed = 37, 45, 2, 8, 12
    sc, cam = _load("cornell_box.json")
    hd = sc.device_scene(0)
    ref_frame, ref = _features(hd, cam, w, h, spp, depth, seed)
    tw, th = tile
    for shards in (2, 3, 5):
        own = _owner(w, h, tw, th, shards)
        sums = []
        for s in range(shards):
            frame, _ = _features(hd, cam, w, h, spp, depth, seed, shards, s, tile)
            assert same(frame[own == s], ref_frame[own == s]), (shards, s)
            assert (frame[own != s] == -1.0).all()
            cnt = api.shard_float4_count(_params(w, h, spp, depth, seed, shards, s, tile), s)
            fptr, fcnt = api.render_device_features(hd)
            assert fcnt == cnt and cnt > 0
            t = torch.as_tensor(api.DevicePointer(fptr, (cnt, 9)), device="cuda").clone()
            host = np.frombuffer(t.cpu().numpy().tobytes(), api.FEATURE_SUMS_DTYPE)
            pad = _padding(w, h, tw, th, shards, s, cnt)
            assert (host["shape"][pad] == -1).all() and (host["pad"] == 0).all()
            for k in ("albedo", "normal", "depth", "hits"):
                assert host[k][pad].tobytes() == np.zeros_like(host[k][pad]).tobytes(), (shards, s, k)
            assert (host["hits"][~pad] <= spp).all()
            sums.append(t)
            with pytest.raises(rt.RtError):   # a shard's features are not delivered whole
                api.render_features(hd)
        out = {"albedo": torch.full((h, w, 3), -1.0, dtype=torch.float64, device="cuda"),
               "normal": torch.full((h, w, 3), -1.0, dtype=torch.float64, device="cuda"),
               "depth": torch.full((h, w), -1.0, dtype=torch.float64, device="cuda"),
               "coverage": torch.full((h, w), -1.0, dtype=torch.float64, device="cuda"),
               "shape": torch.full((h, w), -7, dtype=torch.int32, device="cuda")}
        api.assemble_features(hd, _params(w, h, spp, depth, seed, shards, 0, tile), [s.data_ptr() for s in sums],
                              {k: v.data_ptr() for k, v in out.items()})
        torch.cuda.synchronize()
        assert same_features({k: v.cpu().numpy() for k, v in out.items()}, ref), shards
        # a plane left out is not written
        depth_only = torch.full((h, w), -1.0, dtype=torch.float64, device="cuda")
        api.assemble_features(hd, _params(w, h, spp, depth, seed, shards, 0, tile), [s.data_ptr() for s in sums],
                              {"depth": depth_only.data_ptr()}, stream=torch.cuda.current_stream().cuda_stream or 1)
        torch.cuda.synchronize()
        assert same(depth_only.cpu().numpy(), ref["depth"])


def test_multi_device_handle():
    n_dev = rt.device_count()
    if n_dev < 2:
        pytest.skip("needs at least 2 GPUs")
    w, h, spp, depth, seed = 120, 70, 2, 8, 8
    sc, cam = _load("cornell_box.json")
    ref_frame, ref = _features(sc.device_scene(0), cam, w, h, spp, depth, seed)
    hm = sc.device_scene_multi(list(range(n_dev)))
    for size in ((w, h), (33, 17), (w, h)):   # the staging grows and shrinks between frames
        frame, feats = _features(hm, cam, size[0], size[1], spp, depth, seed)
        want = ref if size == (w, h) else _features(sc.device_scene(0), cam, size[0], size[1], spp, depth, seed)[1]
        assert same_features(feats, want), size
    assert same(frame, ref_frame)
    ren = rt.GpuRenderer(sc, 12, depth, seed=seed, devices=list(range(n_dev)))
    frame, feats = ren.render_features(cam, w, h, spp)
    assert same(frame, ref_frame) and same_features(feats, ref)


def test_renderer_features():
    sc, cam = _load("dupin.json")
    w, h, spp, depth, seed = 24, 16, 2, 6, 4
    ren = rt.GpuRenderer(sc, 12, depth, seed=seed)
    frame, feats = ren.render_features(cam, w, h, spp)
    assert frame.shape == (h, w, 3) and feats["albedo"].shape == (h, w, 3) and feats["shape"].dtype == np.int32
    assert same(frame, ren.render(cam, w, h, spp))
    assert same_features(feats, _replay(sc, cam, w, h, spp, seed))


def test_distributed_renderer_features():
    """DistributedRenderer.render_features under torchrun over every GPU of the box (one rank when there is one)"""
    torch = pytest.importorskip("torch")
    tool = os.path.join(ROOT, "tools", "check_distributed_features.py")
    n = max(1, min(torch.cuda.device_count(), 8))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr",
           "127.0.0.1", "--master-port", "29564", tool]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert r.stdout.count("identical") == 4, r.stdout[-3000:]


# ---- state ---------------------------------------------------------------------------------------------------------

def test_state():
    sc, cam = _load("cornell_box.json")
    hd = sc.device_scene(0)
    w, h, spp, depth, seed = 20, 12, 3, 8, 3
    lib = _ffi.core()
    planes = _ffi.FeaturePlanes()
    ptr, cnt = C.c_void_p(), C.c_uint64()
    state = lambda: (lib.rt_render_features(hd, None, C.byref(planes)),
                     lib.rt_render_device_features(hd, C.byref(ptr), C.byref(cnt)))
    # RT_ERR_STATE before any frame and after plain, adaptive, counts, views and layers frames
    assert state() == (_ffi.RT_ERR_STATE, _ffi.RT_ERR_STATE)
    plain = _plain(hd, cam, w, h, spp, depth, seed)
    assert state() == (_ffi.RT_ERR_STATE, _ffi.RT_ERR_STATE)
    frame, feats = _features(hd, cam, w, h, spp, depth, seed)
    others = [
        lambda: api.render_start_adaptive(hd, cam, api.render_params(w, h, 8, depth, seed), 2, 0.1, 0.0),
        lambda: api.render_start_counts(hd, cam, api.render_params(w, h, 4, depth, seed), np.full((h, w), 2, np.uint32)),
        lambda: api.render_start_views(hd, [cam, cam], api.render_params(w, h, spp, depth, seed)),
        lambda: api.render_start_layers(hd, cam, api.render_params(w, h, spp, depth, seed), 3),
        lambda: api.render_start(hd, cam, api.render_params(w, h, spp, depth, seed)),
    ]
    for start in others:
        _features(hd, cam, w, h, spp, depth, seed)
        start()
        assert state() == (_ffi.RT_ERR_STATE, _ffi.RT_ERR_STATE)
    # after a shard: the sums are there, the whole planes are not
    _features(hd, cam, w, h, spp, depth, seed, 2, 1, (8, 8))
    assert state() == (_ffi.RT_ERR_STATE, _ffi.RT_OK)
    # readable until the next start, as often as asked; paths count as for rt_render_start
    sc.reset_stats(0)
    frame2, feats2 = _features(hd, cam, w, h, spp, depth, seed)
    assert sc.stats(0).paths == w * h * spp
    assert same(frame2, frame) and same_features(feats2, feats) and same_features(api.render_features(hd), feats)
    # a start stops a frame in flight; stop works
    api.render_start_features(hd, cam, api.render_params(w, h, spp, depth, seed))
    api.render_start_features(hd, cam, api.render_params(w, h, 1, depth, seed))
    assert same_features(api.render_features(hd), _replay(sc, cam, w, h, 1, seed))
    api.render_start_features(hd, cam, api.render_params(w, h, spp, depth, seed))
    assert lib.rt_render_stop(hd) == _ffi.RT_OK
    assert state()[0] == _ffi.RT_ERR_STATE
    # an accumulation: a features frame neither continues nor seeds one
    api.render_set_accumulate(hd, True)
    _plain(hd, cam, w, h, spp, depth, seed)
    assert api.render_accumulated_samples(hd) == spp
    again, f3 = _features(hd, cam, w, h, spp, depth, seed)
    assert same(again, plain) and same_features(f3, feats) and api.render_accumulated_samples(hd) == 0
    assert same(_plain(hd, cam, w, h, spp, depth, seed), plain) and api.render_accumulated_samples(hd) == spp
    api.render_set_accumulate(hd, False)
    # pixel stats as after rt_render_start
    _features(hd, cam, w, h, spp, depth, seed)
    counts, moments = api.render_pixel_stats(hd)
    assert (counts == spp).all() and moments is None


def test_features_after_scene_updates_equal_a_fresh_handle():
    sc, cam = _load("cornell_box.json")
    hd = sc.device_scene(0)
    w, h, spp, depth, seed = 20, 14, 2, 8, 6
    _features(hd, cam, w, h, spp, depth, seed)
    ed = Edited(sc)
    rng = np.random.default_rng(4)
    idx = [0, 2, 5]
    inv, dirc = ed.move(rng, idx, 0.2)
    update_transforms(hd, idx, inv, dirc)
    for step in ("transforms", "description"):
        if step == "description":
            ed.move(rng, [1, 3], 0.3)
            api.scene_update(hd, ed.desc())
        frame, feats = _features(hd, cam, w, h, spp, depth, seed)
        fresh = create(ed.desc())
        try:
            ref_frame, ref = _features(fresh, cam, w, h, spp, depth, seed)
        finally:
            _ffi.core().rt_scene_destroy(fresh)
        assert same(frame, ref_frame) and same_features(feats, ref), step


# ---- argument edges ------------------------------------------------------------------------------------------------

def test_argument_edges_keep_the_last_frame():
    sc, cam = _load("spheres.json")
    hd = sc.device_scene(0)
    w, h, spp, depth, seed = 9, 7, 2, 62, 1
    lib = _ffi.core()
    frame, feats = _features(hd, cam, w, h, spp, depth, seed)
    bads = [api.render_params(w, h, spp, 63, seed), api.render_params(0, h, spp, depth, seed),
            api.render_params(w, h, 0, depth, seed), api.render_params(w, h, 0xFFFFFFF1, depth, seed),
            api.render_params(w, h, spp, depth, seed, 17, 0), api.render_params(w, h, spp, depth, seed, 2, 2)]
    huge = api.render_params(1, 0xFFFFFFFF, 1, 8, 0, 2, 0)   # one-row tiles as wide as 2^32 - 1 pixels: sums overflow
    huge.tile_width, huge.tile_height = 0xFFFFFFFF, 1
    for bad in bads + [huge]:
        assert lib.rt_render_start_features(hd, C.byref(cam), C.byref(bad)) == _ffi.RT_ERR_INVALID
        assert same_features(api.render_features(hd), feats)
    assert lib.rt_render_start_features(hd, None, C.byref(bads[0])) == _ffi.RT_ERR_INVALID
    assert same_features(api.render_features(hd), feats)
    ptr, cnt = C.c_void_p(), C.c_uint64()
    assert lib.rt_render_device_frame(hd, C.byref(ptr), C.byref(cnt)) == _ffi.RT_OK and cnt.value == w * h
    assert lib.rt_render_device_features(hd, None, C.byref(cnt)) == _ffi.RT_ERR_INVALID
    assert lib.rt_render_device_features(hd, C.byref(ptr), None) == _ffi.RT_ERR_INVALID


# ---- the oracle ----------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", ["spheres.json", "cornell_box.json", "dupin.json", "4b", "light_source.json"])
def test_spp1_features_against_the_oracle(name):
    """an spp-1 frame's shape, depth and normal are the oracle's nearest hit of the same camera rays, bit for bit (the
    normal as a sum from +0.0: a -0.0 component of the hit's normal reads +0.0)"""
    sc, cam = _load(name)
    w, h, seed = 48, 36, 11
    _, feats = _features(sc.device_scene(0), cam, w, h, 1, 8, seed)
    rays, _ = api.primary_rays(cam, w, h, np.arange(w * h), 1, seed)
    want = po.OracleScene(sc.desc()).intersect_batch(rays)
    hit = want["index"] >= 0
    assert hit.any()
    assert same(feats["shape"].reshape(-1), want["index"])
    assert same(feats["depth"].reshape(-1)[hit], want["t"][hit]) and np.isposinf(feats["depth"].reshape(-1)[~hit]).all()
    assert same(feats["normal"].reshape(-1, 3)[hit], 0.0 + want["normal"][hit])
    assert same(feats["normal"].reshape(-1, 3)[~hit], np.zeros(((~hit).sum(), 3)))
    assert same(feats["coverage"].reshape(-1), hit.astype(np.float64))
