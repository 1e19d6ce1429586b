"""rt_render_start_layers: the rt_render_start frame with each pixel's radiance split by the level that ended its paths.

The frame of a layers frame must be rt_render_start's bit for bit, and every layer must equal, bit for bit, api.layer_means
over api.trace_paths(primary rays, record=True) -- the per-path radiance and ending level of the very paths the frame
traces (trace_paths is pinned to the frame and to the oracle by test_gpu_scatter.py) -- whatever the batch size, the
lanes, the kernel timing, the fused fallback, the devices or the shards.
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

from conftest import scene_path
from test_gpu_frame_edges import _owner, _params, marched_scene
from test_gpu_render import _variant_4b
from test_gpu_scene_update import Edited, create, update_transforms

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCENES = ["spheres.json", "cornell_box.json", "dupin.json", "4b", "light_source.json", "march33"]


def same(a, b):
    """bit for bit, NaN payloads and signed zeros included"""
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.tobytes() == b.tobytes()


def _load(name):
    if name == "march33":   # 33 ray-marched shapes: the fused k_bounce renders it
        sc = rt.Scene.from_json(json.dumps(marched_scene(33)), add_random_spheres=False)
        return sc, sc.camera()
    if name == "4b":
        sc = rt.Scene.from_file(scene_path("detached_materials.json"), random_spheres_seed=1)
        return sc, _variant_4b(sc)
    sc = rt.Scene.from_file(scene_path(name), random_spheres_seed=1)
    return sc, sc.camera()


def _layers(hd, cam, w, h, spp, depth, seed, n_layers, shards=1, index=0, tile=(0, 0)):
    """one layers frame through the raw calls: (frame polled into a buffer of -1, layers) -- layers None for a shard"""
    api.render_start_layers(hd, cam, _params(w, h, spp, depth, seed, shards, index, tile), n_layers)
    frame = np.full((h, w, 3), -1.0)
    while not api.render_poll(hd, frame):
        pass
    return frame, (api.render_layers(hd) if shards == 1 else None)


def _plain(hd, cam, w, h, spp, depth, seed):
    api.render_start(hd, cam, api.render_params(w, h, spp, depth, seed))
    frame = np.zeros((h, w, 3))
    api.render_wait(hd, frame)
    return frame


def _replay(sc, cam, w, h, spp, depth, seed, n_layers_list):
    """the contract restated: the frame's own camera rays through trace_paths, binned by each path's last level"""
    rays, keys = api.primary_rays(cam, w, h, np.arange(w * h), spp, seed)
    L, record = api.trace_paths(sc, rays, keys, depth, seed, record=True)
    levels = api.path_levels(record, len(rays))
    assert (levels >= 0).all() and levels.max() <= depth
    offsets = np.arange(0, w * h * spp + 1, spp)
    return {n: api.layer_means(L, levels, offsets, n).reshape(n, h, w, 3) for n in n_layers_list}, levels


def _layer_counts(depth):
    return sorted({1, 2, 3, depth + 1, 63})


# ---- the contract --------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", SCENES)
def test_layers_replay_trace_paths(name):
    """depths 0, 1, 8, 62 and seeds 0, 2^64-1: the frame is rt_render_start's, layer 0 of one layer is the frame, and
    every layer of 1, 2, 3, depth + 1 and 63 layers is layer_means over trace_paths, bit for bit"""
    w, h, spp = 14, 10, 3
    sc, cam = _load(name)
    hd = sc.device_scene(0)
    for seed in (0, (1 << 64) - 1):
        for depth in (0, 1, 8, 62):
            counts = _layer_counts(depth)
            want, levels = _replay(sc, cam, w, h, spp, depth, seed, counts)
            plain = _plain(hd, cam, w, h, spp, depth, seed)
            for n in counts:
                frame, layers = _layers(hd, cam, w, h, spp, depth, seed, n)
                assert same(frame, plain), (name, seed, depth, n)
                assert same(layers, want[n]), (name, seed, depth, n)
                if n == 1:
                    assert same(layers[0], frame)
                if n > depth + 1:   # layers above max_depth are zero
                    assert same(layers[depth + 1:], np.zeros_like(layers[depth + 1:]))
            # a pixel whose samples all end on one level has that layer equal to its frame pixel
            lv = levels.reshape(h * w, spp)
            one = (lv == lv[:, :1]).all(axis=1)
            layers = want[63].reshape(63, h * w, 3)
            for p in np.flatnonzero(one):
                assert same(layers[lv[p, 0], p], frame.reshape(-1, 3)[p])


def test_layers_add_up_to_the_frame():
    """the layers of a deep frame add up to the frame within the reassociation of its f64 sums"""
    sc, cam = _load("cornell_box.json")
    hd = sc.device_scene(0)
    w, h, spp, depth = 64, 48, 16, 50
    for n in (4, 51, 63):
        frame, layers = _layers(hd, cam, w, h, spp, depth, 7, n)
        bound = (n + spp) * 2.0 ** -52 * np.abs(layers).sum(0) + 1e-300
        assert (np.abs(layers.sum(0) - frame) <= bound).all(), n
        assert (layers >= 0).all()


# ---- schedules -----------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", ["cornell_box.json", "march33"])
def test_schedules_give_the_same_layers(monkeypatch, name):
    """batches of 1 and 7 paths and of one pixel's paths - 1 / + 1, 1 / 2 / 3 lanes, kernel timing, the fused k_bounce"""
    w, h, spp, depth, seed, n = 16, 12, 5, 8, 21, 4
    sc, cam = _load(name)
    ref_frame, ref = _layers(sc.device_scene(0), cam, w, h, spp, depth, seed, n)

    def run(env, timing=False):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        alt, _ = _load(name)   # a new device handle reads the variables
        hd = alt.device_scene(0)
        if timing:
            alt.set_kernel_timing(True, 0)
        out = _layers(hd, cam, w, h, spp, depth, seed, n)
        if timing:
            s = alt.stats(0)
            assert s.ms_resolve > 0 and s.launches_extend > 0
        for k in env:
            monkeypatch.delenv(k)
        return out

    for env in ({"RT_B200_BATCH_PATHS": "1"}, {"RT_B200_BATCH_PATHS": "7"},
                {"RT_B200_BATCH_PATHS": str(spp - 1)}, {"RT_B200_BATCH_PATHS": str(spp + 1)},
                {"RT_B200_BATCH_PATHS": "100", "RT_B200_LANES": "1"},
                {"RT_B200_BATCH_PATHS": "100", "RT_B200_LANES": "2"}, {"RT_B200_BATCH_PATHS": "100", "RT_B200_LANES": "3"},
                {"RT_B200_FUSED_BOUNCE": "1"}, {"RT_B200_FUSED_BOUNCE": "1", "RT_B200_BATCH_PATHS": "7"}):
        frame, layers = run(env)
        assert same(frame, ref_frame) and same(layers, ref), env
    frame, layers = run({"RT_B200_BATCH_PATHS": "7"}, timing=True)
    assert same(frame, ref_frame) and same(layers, ref)


# ---- images --------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("w,h", [(1, 1), (1, 45), (45, 1), (2, 70000)])
def test_image_shapes(w, h):
    sc, cam = _load("spheres.json")
    hd = sc.device_scene(0)
    spp, depth, seed, n = (1, 4, 9, 3) if w * h > 1000 else (4, 8, 9, 5)
    want, _ = _replay(sc, cam, w, h, spp, depth, seed, [n])
    frame, layers = _layers(hd, cam, w, h, spp, depth, seed, n)
    ptr, count = api.render_layers(hd, device=True)
    assert count == n * w * h and ptr
    assert same(layers, want[n])
    assert same(frame, _plain(hd, cam, w, h, spp, depth, seed))


# ---- devices and shards --------------------------------------------------------------------------------------------

@pytest.mark.parametrize("tile", [(16, 16), (32, 32)])
def test_explicit_shards_assemble_to_the_layers(tile):
    """shards 2, 4, 8, 16 (clipped border tiles): each shard's polled pixels are the frame's, and rt_assemble_layers over
    the gathered accumulators and layer sums is the unsharded layers frame bit for bit"""
    torch = pytest.importorskip("torch")
    w, h, spp, depth, seed, n = 37, 45, 2, 8, 12, 4
    sc, cam = _load("cornell_box.json")
    hd = sc.device_scene(0)
    ref_frame, ref = _layers(hd, cam, w, h, spp, depth, seed, n)
    tw, th = tile
    for shards in (2, 4, 8, 16):
        own = _owner(w, h, tw, th, shards)
        accs, sums = [], []
        for s in range(shards):
            frame, _ = _layers(hd, cam, w, h, spp, depth, seed, n, shards, s, tile)
            assert same(frame[own == s], ref_frame[own == s]), (shards, s)
            assert (frame[own != s] == -1.0).all()
            cnt = api.shard_float4_count(_params(w, h, spp, depth, seed, shards, s, tile), s)
            aptr, acnt = api.render_device_result(hd)
            lptr, lcnt = api.render_device_layers(hd)
            assert acnt == cnt and lcnt == n * cnt
            if cnt == 0:   # (a shard without tiles: never read)
                accs.append(torch.zeros((1, 4), dtype=torch.float64, device="cuda"))
                sums.append(torch.zeros((1, 3), dtype=torch.float64, device="cuda"))
                continue
            accs.append(torch.as_tensor(api.DevicePointer(aptr, (cnt, 4)), device="cuda").clone())
            sums.append(torch.as_tensor(api.DevicePointer(lptr, (n * cnt, 3)), device="cuda").clone())
            # a shard's layers are not delivered whole: rt_render_layers refuses
            with pytest.raises(rt.RtError):
                api.render_layers(hd)
        out = torch.full((n, h, w, 3), -1.0, dtype=torch.float64, device="cuda")
        api.assemble_layers(hd, _params(w, h, spp, depth, seed, shards, 0, tile), n, [a.data_ptr() for a in accs],
                            [s.data_ptr() for s in sums], out.data_ptr())
        torch.cuda.synchronize()
        assert same(out.cpu().numpy(), ref), shards


def test_multi_device_handle():
    n_dev = rt.device_count()
    if n_dev < 2:
        pytest.skip("needs at least 2 GPUs")
    w, h, spp, depth, seed, n = 120, 70, 2, 8, 8, 5
    sc, cam = _load("cornell_box.json")
    ref_frame, ref = _layers(sc.device_scene(0), cam, w, h, spp, depth, seed, n)
    hm = sc.device_scene_multi(list(range(n_dev)))
    for n_layers in (n, 63, 2):   # the staging grows and shrinks between frames
        frame, layers = _layers(hm, cam, w, h, spp, depth, seed, n_layers)
        assert same(frame, ref_frame)
        want = ref if n_layers == n else _layers(sc.device_scene(0), cam, w, h, spp, depth, seed, n_layers)[1]
        assert same(layers, want), n_layers
    ren = rt.GpuRenderer(sc, 12, depth, seed=seed, devices=list(range(n_dev)))
    frame, layers = ren.render_layers(cam, w, h, spp, n)
    assert same(frame, ref_frame) and same(layers, ref)


def test_renderer_layers():
    sc, cam = _load("dupin.json")
    w, h, spp, depth, seed = 24, 16, 2, 6, 4
    ren = rt.GpuRenderer(sc, 12, depth, seed=seed)
    frame, layers = ren.render_layers(cam, w, h, spp, 3)
    assert frame.shape == (h, w, 3) and layers.shape == (3, h, w, 3) and layers.dtype == np.float64
    assert same(frame, ren.render(cam, w, h, spp))
    want, _ = _replay(sc, cam, w, h, spp, depth, seed, [3])
    assert same(layers, want[3])


def test_distributed_renderer_layers():
    """DistributedRenderer.render_layers under torchrun over every GPU of the box (one rank when there is one)"""
    torch = pytest.importorskip("torch")
    tool = os.path.join(ROOT, "tools", "check_distributed_layers.py")
    n = max(1, min(torch.cuda.device_count(), 8))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr",
           "127.0.0.1", "--master-port", "29563", tool]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert r.stdout.count("identical") == 4, r.stdout[-3000:]


# ---- state ---------------------------------------------------------------------------------------------------------

def test_state():
    sc, cam = _load("cornell_box.json")
    hd = sc.device_scene(0)
    w, h, spp, depth, seed = 20, 12, 3, 8, 3
    lib = _ffi.core()
    ptr, cnt = C.c_void_p(), C.c_uint64()
    # RT_ERR_STATE before any frame and after a plain one
    assert lib.rt_render_layers(hd, None, C.byref(ptr), C.byref(cnt)) == _ffi.RT_ERR_STATE
    plain = _plain(hd, cam, w, h, spp, depth, seed)
    assert lib.rt_render_layers(hd, None, C.byref(ptr), C.byref(cnt)) == _ffi.RT_ERR_STATE
    assert lib.rt_render_device_layers(hd, C.byref(ptr), C.byref(cnt)) == _ffi.RT_ERR_STATE
    # paths count as for rt_render_start; a start stops a frame in flight; stop works
    sc.reset_stats(0)
    frame, layers = _layers(hd, cam, w, h, spp, depth, seed, 4)
    assert sc.stats(0).paths == w * h * spp
    api.render_start_layers(hd, cam, api.render_params(w, h, spp, depth, seed), 4)
    api.render_start_layers(hd, cam, api.render_params(w, h, spp, depth, seed), 2)   # stops the first
    two = api.render_layers(hd)
    assert two.shape == (2, h, w, 3) and same(two[0], layers[0])
    api.render_start_layers(hd, cam, api.render_params(w, h, spp, depth, seed), 4)
    assert lib.rt_render_stop(hd) == _ffi.RT_OK
    assert lib.rt_render_layers(hd, None, C.byref(ptr), C.byref(cnt)) == _ffi.RT_ERR_STATE
    # an accumulation afterwards starts afresh, and a layers frame neither continues nor seeds one
    api.render_set_accumulate(hd, True)
    _plain(hd, cam, w, h, spp, depth, seed)
    assert api.render_accumulated_samples(hd) == spp
    again, _ = _layers(hd, cam, w, h, spp, depth, seed, 3)
    assert same(again, plain) and api.render_accumulated_samples(hd) == 0
    assert same(_plain(hd, cam, w, h, spp, depth, seed), plain) and api.render_accumulated_samples(hd) == spp
    api.render_set_accumulate(hd, False)
    # pixel stats as after rt_render_start
    _layers(hd, cam, w, h, spp, depth, seed, 3)
    counts, moments = api.render_pixel_stats(hd)
    assert (counts == spp).all() and moments is None


def test_layers_after_a_transforms_update_equal_a_fresh_handle():
    sc, cam = _load("cornell_box.json")
    hd = sc.device_scene(0)
    w, h, spp, depth, seed, n = 20, 14, 2, 8, 6, 5
    _layers(hd, cam, w, h, spp, depth, seed, n)
    ed = Edited(sc)
    idx = [0, 2, 5]
    inv, dirc = ed.move(np.random.default_rng(4), idx, 0.2)
    update_transforms(hd, idx, inv, dirc)
    frame, layers = _layers(hd, cam, w, h, spp, depth, seed, n)
    fresh = create(ed.desc())
    try:
        ref_frame, ref = _layers(fresh, cam, w, h, spp, depth, seed, n)
    finally:
        _ffi.core().rt_scene_destroy(fresh)
    assert same(frame, ref_frame) and same(layers, ref)


# ---- argument edges ------------------------------------------------------------------------------------------------

def test_argument_edges_keep_the_last_frame():
    sc, cam = _load("spheres.json")
    hd = sc.device_scene(0)
    w, h, spp, depth, seed = 9, 7, 2, 62, 1
    lib = _ffi.core()
    frame, layers = _layers(hd, cam, w, h, spp, depth, seed, 63)
    assert layers.shape == (63, h, w, 3)
    p = api.render_params(w, h, spp, depth, seed)
    for bad in (0, 64):
        assert lib.rt_render_start_layers(hd, C.byref(cam), C.byref(p), bad) == _ffi.RT_ERR_INVALID
    bad_p = api.render_params(w, h, spp, 63, seed)   # max_depth above 62
    assert lib.rt_render_start_layers(hd, C.byref(cam), C.byref(bad_p), 3) == _ffi.RT_ERR_INVALID
    assert same(api.render_layers(hd), layers)
    ptr, cnt = C.c_void_p(), C.c_uint64()
    assert lib.rt_render_device_frame(hd, C.byref(ptr), C.byref(cnt)) == _ffi.RT_OK and cnt.value == w * h
    # a layer buffer whose size overflows: a 1-pixel-wide image with tall tiles pads every shard enormously
    huge = api.render_params(0xFFFFFFFF, 1, 1, 8, 0, 2, 0)
    huge.tile_width, huge.tile_height = 1, 0xFFFFFFFF
    assert lib.rt_render_start_layers(hd, C.byref(cam), C.byref(huge), 63) == _ffi.RT_ERR_INVALID
    assert same(api.render_layers(hd), layers)
