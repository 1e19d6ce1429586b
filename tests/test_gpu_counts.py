"""rt_render_start_counts: frames with the caller's sample count per pixel.

Every pixel of a counts frame must equal, bit for bit, the rt_render_start pixel at its count -- i.e.
trace_pixel_samples_group over its first counts[p] camera rays -- whatever the batch size, the lanes, the kernel timing,
the fused fallback, the devices or the shards; a count-0 pixel is NaN.
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
from test_gpu_adaptive import _variant_4b
from test_gpu_frame_edges import _device_accum, _owner, _params, check_pixels, marched_scene

pytestmark = pytest.mark.gpu

DEPTH = 8
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _load(name, variant=""):
    if name == "march33":
        sc = rt.Scene.from_json(json.dumps(marched_scene(33)), add_random_spheres=False)
        return sc, sc.camera()
    sc = rt.Scene.from_file(scene_path(name), random_spheres_seed=1)
    return sc, (_variant_4b(sc) if variant == "4b" else sc.camera())


def _counts(hd, cam, counts, depth=DEPTH, seed=5, cap=None, shards=1, index=0, tile=(0, 0), fill=0.0):
    """one counts frame through the raw calls, waited for into a buffer of `fill`"""
    h, w = counts.shape
    cap = cap or max(int(counts.max()), 1)
    api.render_start_counts(hd, cam, _params(w, h, cap, depth, seed, shards, index, tile), counts)
    out = np.full((h, w, 3), fill)
    api.render_wait(hd, out)
    return out


def _uniform(hd, cam, w, h, spp, depth=DEPTH, seed=5):
    api.render_start(hd, cam, api.render_params(w, h, spp, depth, seed))
    out = np.zeros((h, w, 3))
    api.render_wait(hd, out)
    return out


def _by_uniform(hd, cam, counts, depth=DEPTH, seed=5):
    """what the contract says: pixel p of the rt_render_start frame at samples_number = counts[p]; NaN at count 0"""
    h, w = counts.shape
    ref = np.full((h, w, 3), np.nan)
    for k in np.unique(counts):
        if k:
            sel = counts == k
            ref[sel] = _uniform(hd, cam, w, h, int(k), depth, seed)[sel]
    return ref


def _count_rays(cam, w, h, counts, seed):
    """the first counts[p] camera rays of every pixel (MultisamplerRayCaster::next with the Philox draws of event 0) as
    trace_pixel_samples_group's groups"""
    flat = counts.reshape(-1)
    rays = np.empty((int(flat.sum()), 6))
    k = 0
    for p in np.flatnonzero(flat):
        x, y = int(p % w), int(p // w)
        for s in range(int(flat[p])):
            u, v = po.philox_stream(seed, int(p), s, 0, 2)
            rays[k] = po.get_ray(cam, w, h, x + u, y + v)
            k += 1
    offsets = np.concatenate([[0], np.cumsum(flat, dtype=np.uint64)]).astype(np.uint64)
    return rays, offsets, np.arange(w * h, dtype=np.uint32)


def _random_map(seed, h, w, hi):
    return np.random.default_rng(seed).integers(0, hi + 1, (h, w)).astype(np.uint32)


# ---- the frame ---------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name,variant", [("spheres.json", ""), ("cornell_box.json", ""), ("dupin.json", ""),
                                          ("detached_materials.json", "4b")])
def test_uniform_map_is_the_frame(name, variant):
    w, h, spp = 64, 48, 4
    sc, cam = _load(name, variant)
    hd = sc.device_scene(0)
    ref = _uniform(hd, cam, w, h, spp)
    assert np.array_equal(_counts(hd, cam, np.full((h, w), spp, np.uint32)), ref)
    # the cap may exceed every count
    assert np.array_equal(_counts(hd, cam, np.full((h, w), spp, np.uint32), cap=1000), ref)


def test_random_map():
    """counts 0..64 at 160x120: every pixel == trace_pixel_samples_group over its first counts[p] camera rays == the
    uniform frame of its count, and within one float ulp per path of the oracle; count 0 is NaN; paths == sum of the
    counts; pixel stats == the map; the device tone map == rt_tonemap_rgba8 of the frame"""
    w, h, seed = 160, 120, 9
    sc, cam = _load("spheres.json")
    hd = sc.device_scene(0)
    counts = _random_map(3, h, w, 64)
    sc.reset_stats(0)
    frame = _counts(hd, cam, counts, seed=seed)
    assert sc.stats(0).paths == int(counts.sum(dtype=np.uint64))
    assert np.isnan(frame[counts == 0]).all() and np.isfinite(frame[counts > 0]).all()
    got_counts, moments = api.render_pixel_stats(hd)
    assert np.array_equal(got_counts, counts) and moments is None
    assert _ffi.core().rt_render_pixel_stats(hd, None, np.empty((h, w, 2)).ctypes.data_as(C.c_void_p)) == _ffi.RT_ERR_STATE
    assert np.array_equal(api.tonemap_last_frame(hd).reshape(h, w, 4), rt.tonemap_rgba8(sc, frame))

    rays, offsets, pix = _count_rays(cam, w, h, counts, seed)
    groups = sc.trace_pixel_samples_group(rays, offsets, pix, DEPTH, seed=seed)
    assert np.array_equal(groups.reshape(h, w, 3), frame, equal_nan=True)
    assert np.array_equal(_by_uniform(hd, cam, counts, seed=seed), frame, equal_nan=True)

    osc = po.OracleScene(sc.desc())
    sample = np.sort(np.random.default_rng(4).choice(w * h, 600, replace=False))
    flat_counts, flat = counts.reshape(-1), frame.reshape(-1, 3)
    for k in np.unique(flat_counts[sample]):
        if k:
            pixels = sample[flat_counts[sample] == k]
            cols = osc.frame_sample_colors(cam, w, h, int(k), DEPTH, seed, pixels=pixels)
            check_pixels(flat[pixels], cols, f"count {k}")


@pytest.mark.parametrize("name,rel", [("cornell_box.json", 0.05), ("spheres.json", 0.02)])
def test_adaptive_replay(name, rel):
    """the counts an adaptive frame ends with give that adaptive frame back, bit for bit"""
    w, h, spp, mn, seed = 96, 72, 64, 4, 5
    sc, cam = _load(name)
    hd = sc.device_scene(0)
    api.render_start_adaptive(hd, cam, api.render_params(w, h, spp, DEPTH, seed), mn, rel, 0.0)
    adaptive = np.zeros((h, w, 3))
    api.render_wait(hd, adaptive)
    counts, _ = api.render_pixel_stats(hd)
    assert len(np.unique(counts)) > 1
    assert np.array_equal(_counts(hd, cam, counts, seed=seed, cap=spp), adaptive)
    ren = rt.GpuRenderer(sc, 12, DEPTH, seed=seed)
    assert np.array_equal(ren.render_counts(cam, counts), adaptive)


# ---- schedules ---------------------------------------------------------------------------------------------------

def test_schedules_give_the_same_frame(monkeypatch):
    """batches of 1 and 7 paths and just below and above the largest pixel's count (pixels cut over batches and over
    pieces), 1 / 2 / 3 lanes, kernel timing on, the fused k_bounce: the same frame, bit for bit, also when polled"""
    w, h, seed = 16, 12, 21
    counts = _random_map(5, h, w, 8)
    counts[3, 4] = 50
    counts[0, 0] = 0
    counts[h - 1, w - 1] = 17
    sc, cam = _load("spheres.json")
    ref = _counts(sc.device_scene(0), cam, counts, seed=seed)
    assert np.array_equal(_by_uniform(sc.device_scene(0), cam, counts, seed=seed), ref, equal_nan=True)

    def run(env, timing=False):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        alt, _ = _load("spheres.json")   # a new device handle reads the variables
        hd = alt.device_scene(0)
        if timing:
            alt.set_kernel_timing(True, 0)
        api.render_start_counts(hd, cam, api.render_params(w, h, 50, DEPTH, seed), counts)
        buf = np.full((h, w, 3), -1.0)
        while not api.render_poll(hd, buf):
            pass
        if timing:
            s = alt.stats(0)
            assert s.ms_raygen > 0 and s.ms_resolve > 0 and s.launches_extend > 0
        for k in env:
            monkeypatch.delenv(k)
        return buf

    for env in ({"RT_B200_BATCH_PATHS": "1"}, {"RT_B200_BATCH_PATHS": "7"}, {"RT_B200_BATCH_PATHS": "49"},
                {"RT_B200_BATCH_PATHS": "51"}, {"RT_B200_BATCH_PATHS": "100", "RT_B200_LANES": "1"},
                {"RT_B200_BATCH_PATHS": "100", "RT_B200_LANES": "2"}, {"RT_B200_BATCH_PATHS": "100", "RT_B200_LANES": "3"},
                {"RT_B200_FUSED_BOUNCE": "1"}, {"RT_B200_FUSED_BOUNCE": "1", "RT_B200_BATCH_PATHS": "7"}):
        assert np.array_equal(run(env), ref, equal_nan=True), env
    assert np.array_equal(run({"RT_B200_BATCH_PATHS": "7"}, timing=True), ref, equal_nan=True)


def test_fused_fallback_scene():
    """33 marched shapes (the fused fallback by scene): every pixel == trace_pixel_samples_group over its camera rays"""
    w, h, seed = 16, 12, 3
    counts = _random_map(6, h, w, 4)
    sc, cam = _load("march33")
    frame = _counts(sc.device_scene(0), cam, counts, seed=seed)
    rays, offsets, pix = _count_rays(cam, w, h, counts, seed)
    groups = sc.trace_pixel_samples_group(rays, offsets, pix, DEPTH, seed=seed)
    assert np.array_equal(groups.reshape(h, w, 3), frame, equal_nan=True)


# ---- devices and shards ------------------------------------------------------------------------------------------

@pytest.mark.parametrize("tile", [(7, 5), (16, 16)])
def test_explicit_shards_assemble_to_the_frame(tile):
    """shards 2, 4, 8 and 16 with tiles that clip at the border (more shards than tiles included): each shard's polled
    pixels, and rt_assemble_frame over the gathered accumulators, are the unsharded frame bit for bit"""
    torch = pytest.importorskip("torch")
    w, h, seed = 37, 23, 12
    counts = _random_map(7, h, w, 6)
    sc, cam = _load("spheres.json")
    hd = sc.device_scene(0)
    ref = _counts(hd, cam, counts, seed=seed)
    tw, th = tile
    sentinel = torch.full((tw * th, 4), float("nan"), dtype=torch.float64, device="cuda")
    for shards in (2, 4, 8, 16):
        own = _owner(w, h, tw, th, shards)
        accs = []
        for s in range(shards):
            p = _params(w, h, 6, DEPTH, seed, shards, s, tile)
            n = api.shard_float4_count(p, s)
            buf = np.full((h, w, 3), -1.0)
            api.render_start_counts(hd, cam, p, counts)
            while not api.render_poll(hd, buf):
                pass
            assert np.array_equal(buf[own == s], ref[own == s], equal_nan=True), (shards, s)
            assert (buf[own != s] == -1.0).all(), (shards, s)
            acc = _device_accum(torch, hd, n)
            accs.append(acc if acc is not None else sentinel)
        out = torch.full((h, w, 3), -1.0, dtype=torch.float64, device="cuda")
        api.assemble_frame(hd, _params(w, h, 6, DEPTH, seed, shards, 0, tile), [a.data_ptr() for a in accs], out.data_ptr())
        torch.cuda.synchronize()
        assert np.array_equal(out.cpu().numpy(), ref, equal_nan=True), shards


def test_multi_device_handle():
    n = rt.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    w, h, seed = 200, 130, 8
    counts = _random_map(8, h, w, 12)
    sc, cam = _load("cornell_box.json")
    ref = _counts(sc.device_scene(0), cam, counts, seed=seed)
    hm = sc.device_scene_multi(list(range(n)))
    assert np.array_equal(_counts(hm, cam, counts, seed=seed), ref, equal_nan=True)
    ren = rt.GpuRenderer(sc, 12, DEPTH, seed=seed, devices=list(range(n)))
    assert np.array_equal(ren.render_counts(cam, counts), ref, equal_nan=True)


def test_distributed_renderer_with_counts():
    """DistributedRenderer.render(counts=...) under torchrun over every GPU of the box (one rank when there is one)"""
    torch = pytest.importorskip("torch")
    tool = os.path.join(ROOT, "tools", "check_distributed_counts.py")
    n = max(1, min(torch.cuda.device_count(), 8))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr",
           "127.0.0.1", "--master-port", "29561", tool]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert r.stdout.count("identical") == 3, r.stdout[-3000:]


# ---- edges -------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("w,h", [(1, 1), (1, 45), (45, 1), (2, 70000)])
def test_image_shapes(w, h):
    sc, cam = _load("spheres.json")
    hd = sc.device_scene(0)
    counts = _random_map(w * 7 + h, h, w, 3)
    counts.reshape(-1)[0] = 2
    assert np.array_equal(_counts(hd, cam, counts, depth=4), _by_uniform(hd, cam, counts, depth=4), equal_nan=True)


@pytest.mark.parametrize("depth", [0, 1, 62])
def test_depths(depth):
    sc, cam = _load("cornell_box.json")
    hd = sc.device_scene(0)
    counts = _random_map(depth, 24, 32, 5)
    assert np.array_equal(_counts(hd, cam, counts, depth=depth), _by_uniform(hd, cam, counts, depth=depth), equal_nan=True)


@pytest.mark.parametrize("seed", [0, (1 << 64) - 1])
def test_seeds(seed):
    sc, cam = _load("spheres.json")
    hd = sc.device_scene(0)
    counts = _random_map(11, 24, 32, 5)
    assert np.array_equal(_counts(hd, cam, counts, seed=seed), _by_uniform(hd, cam, counts, seed=seed), equal_nan=True)


def test_all_zero_map_and_one_pixel_with_every_sample():
    sc, cam = _load("spheres.json")
    hd = sc.device_scene(0)
    w, h = 40, 30
    zero = np.zeros((h, w), np.uint32)
    sc.reset_stats(0)
    assert np.isnan(_counts(hd, cam, zero)).all()
    assert sc.stats(0).paths == 0
    assert np.array_equal(api.render_pixel_stats(hd)[0], zero)
    assert np.isnan(rt.GpuRenderer(sc, 12, DEPTH, seed=5).render_counts(cam, zero)).all()
    one = zero.copy()
    one[17, 23] = 3000
    frame = _counts(hd, cam, one)
    assert np.isnan(frame[one == 0]).all()
    assert np.array_equal(frame[17, 23], _uniform(hd, cam, w, h, 3000)[17, 23])


def test_handle_reused_across_map_sizes():
    sc, cam = _load("spheres.json")
    hd = sc.device_scene(0)
    for w, h, hi in ((64, 48, 6), (8, 6, 3), (100, 70, 2), (64, 48, 6)):
        counts = _random_map(w + h, h, w, hi)
        fresh, _ = _load("spheres.json")
        assert np.array_equal(_counts(hd, cam, counts), _counts(fresh.device_scene(0), cam, counts), equal_nan=True)


# ---- state -------------------------------------------------------------------------------------------------------

def test_state(monkeypatch):
    """a poll before completion leaves unfinished pixels untouched; stop drains the frame; an accumulating frame after a
    counts frame starts afresh"""
    monkeypatch.setenv("RT_B200_BATCH_PATHS", "2000")
    sc, cam = _load("cornell_box.json")
    hd = sc.device_scene(0)
    w, h = 80, 60
    counts = _random_map(12, h, w, 40)
    ref = _counts(hd, cam, counts)
    api.render_start_counts(hd, cam, api.render_params(w, h, 40, DEPTH, 5), counts)
    buf = np.full((h, w, 3), -7.0)
    first = api.render_poll(hd, buf)
    untouched = (buf == -7.0).all(axis=2)
    assert np.array_equal(buf[~untouched], ref[~untouched], equal_nan=True)
    polls = 1
    while not first and not api.render_poll(hd, buf):
        polls += 1
    assert np.array_equal(buf, ref, equal_nan=True)

    api.render_start_counts(hd, cam, api.render_params(w, h, 40, DEPTH, 5), counts)
    assert _ffi.core().rt_render_stop(hd) == _ffi.RT_OK
    with pytest.raises(rt.RtError):
        api.render_poll(hd, buf)

    api.render_set_accumulate(hd, True)
    a = _uniform(hd, cam, w, h, 4)
    assert api.render_accumulated_samples(hd) == 4
    _counts(hd, cam, counts)
    assert api.render_accumulated_samples(hd) == 0
    assert np.array_equal(_uniform(hd, cam, w, h, 4), a)
    assert api.render_accumulated_samples(hd) == 4
    api.render_set_accumulate(hd, False)


# ---- rejections --------------------------------------------------------------------------------------------------

def test_bad_input_is_rejected():
    sc, cam = _load("spheres.json")
    hd = sc.device_scene(0)
    w, h = 8, 6
    counts = np.full((h, w), 4, np.uint32)
    ptr = counts.ctypes.data_as(C.c_void_p)
    lib = _ffi.core()

    def start(p, c=ptr):
        return lib.rt_render_start_counts(hd, C.byref(cam), C.byref(p), c)

    assert start(api.render_params(w, h, 4, DEPTH), None) == _ffi.RT_ERR_INVALID        # NULL map
    assert start(api.render_params(w, h, 3, DEPTH)) == _ffi.RT_ERR_INVALID              # a count above the cap
    assert start(api.render_params(w, h, 0, DEPTH)) == _ffi.RT_ERR_INVALID              # cap 0
    assert start(api.render_params(w, h, 4, 63)) == _ffi.RT_ERR_INVALID                 # depth 63
    assert start(api.render_params(w, h, 4, DEPTH, 0, 4, 4)) == _ffi.RT_ERR_INVALID     # shard_index >= shard_count
    assert start(api.render_params(w, h, 4, DEPTH, 0, 17, 0)) == _ffi.RT_ERR_INVALID    # more than 16 shards
    for bad in (counts.astype(np.int32), counts.T.copy(), counts.reshape(-1), counts.astype(np.uint64)):
        with pytest.raises(ValueError):
            api.render_start_counts(hd, cam, api.render_params(w, h, 4, DEPTH), bad)
    # the handle is unharmed
    assert np.array_equal(_counts(hd, cam, counts), _uniform(hd, cam, w, h, 4))
