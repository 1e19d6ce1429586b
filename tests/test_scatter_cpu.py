"""Scatter queries (rt_scatter_batch[_device]) without a CUDA device: the core has no CPU fallback, so both entries fail
loudly; the argument checks, api.group_means and the oracle's one-level scatter need no device.

The oracle's scatter is pinned to the oracle itself: iterating it over the levels and folding the colours backwards,
L = a0 * (a1 * (... * last)) as the recursion multiplies, gives orc_groups_sample_colors bit for bit."""
import ctypes as C
import math

import numpy as np
import pytest

import rs_pathtracing_b200 as rt
from rs_pathtracing_b200 import _ffi, api
from oracle import pyoracle as po

from conftest import scene_path
import scatter_oracle


@pytest.mark.skipif(rt.device_count() > 0, reason="checks the behaviour without a CUDA device")
def test_scatter_fails_loudly_without_gpu():
    sc = rt.Scene.from_file(scene_path("cube_test.json"), add_random_spheres=False)
    with pytest.raises(rt.RtError, match="no CUDA device"):
        sc.scatter(np.zeros((1, 6)), np.zeros((1, 2), np.uint32), 0)
    with pytest.raises(rt.RtError, match="no CUDA device"):
        api.trace_paths(sc, np.zeros((3, 6)), np.zeros((3, 2), np.uint32), 4)
    # the device form needs a handle, and no handle can exist without a device
    out = C.c_void_p()
    assert _ffi.core().rt_scene_create(C.byref(sc.desc()), 0, C.byref(out)) == _ffi.RT_ERR_NO_DEVICE


def test_invalid_arguments_in_order():
    """NULL scene, unknown mode, level above 62 -- in that order, before n = 0 -- then NULL rays / keys"""
    lib = _ffi.core()
    rays = np.zeros((4, 6))
    keys = np.zeros((4, 2), np.uint32)
    outs = [np.zeros(4, np.int32), np.zeros(4), np.zeros(4, np.uint8), np.zeros((4, 3)), np.zeros((4, 6))]
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    F = rt.RT_ISECT_FAST
    for fn, extra in ((lib.rt_scatter_batch, ()), (lib.rt_scatter_batch_device, (None,))):
        call = lambda sc, r, k, n, level, mode: fn(sc, r, k, n, level, 0, 0.001, math.inf, mode, *map(p, outs), *extra)
        for args in ((None, p(rays), p(keys), 4, 0, F), (None, p(rays), p(keys), 0, 0, F), (None, None, None, 4, 63, 7)):
            assert call(*args) == _ffi.RT_ERR_INVALID
            assert b"null scene" in lib.rt_last_error()
        assert fn(None, None, None, 0, 0, 0, 0.001, math.inf, F, None, None, None, None, None, *extra) == \
            _ffi.RT_ERR_INVALID


def test_inputs_are_checked_before_the_call():
    sc = rt.Scene.from_file(scene_path("cube_test.json"), add_random_spheres=False)
    rays = np.zeros((6, 6))
    keys = np.zeros((6, 2), np.uint32)
    bad_keys = [np.zeros((6, 2), np.int32), np.zeros((6, 2), np.uint64), np.zeros((5, 2), np.uint32),
                np.zeros((6, 3), np.uint32), np.zeros(12, np.uint32), np.zeros((2, 6), np.uint32).T,
                np.zeros((6, 4), np.uint32)[:, ::2], [[0, 0]] * 6]
    for k in bad_keys:
        with pytest.raises(ValueError):
            sc.scatter(rays, k, 0)
    bad_rays = [np.zeros((6, 3)), np.zeros(36), np.zeros((6, 7)), np.zeros((6, 6), np.float32),
                np.zeros((6, 12))[:, ::2], np.zeros((1, 6, 6)), [[0.0] * 6] * 6]
    for r in bad_rays:
        with pytest.raises(ValueError):
            sc.scatter(r, keys, 0)
    with pytest.raises(ValueError):
        api.trace_paths(sc, rays, keys, 63)
    with pytest.raises(ValueError):
        api.trace_paths(sc, rays, keys, -1)
    api.check_scatter_inputs(rays, keys)


def test_device_form_checks_its_tensors():
    torch = pytest.importorskip("torch")
    sc = rt.Scene.from_file(scene_path("cube_test.json"), add_random_spheres=False)
    rays = torch.zeros((4, 6), dtype=torch.float64)   # host tensors: rejected before any device work
    keys = torch.zeros((4, 2), dtype=torch.uint32)
    with pytest.raises(ValueError):
        sc.scatter(rays, keys, 0)
    with pytest.raises(ValueError):
        sc.scatter(rays, np.zeros((4, 2), np.uint32), 0)


def test_group_means_against_a_loop():
    rng = np.random.default_rng(5)
    sizes = [0, 1, 3, 0, 17, 2, 0, 40, 1]
    n = sum(sizes)
    rad = (rng.normal(size=(n, 3)) * rng.choice([1e-3, 1.0, 1e4], (n, 1))).astype(np.float32)
    rad[5, 1] = np.inf
    offsets = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    got = api.group_means(rad, offsets)
    assert got.shape == (len(sizes), 3) and got.dtype == np.float64
    for g in range(len(sizes)):
        a, b = int(offsets[g]), int(offsets[g + 1])
        if a == b:
            assert np.isnan(got[g]).all()
            continue
        s = [0.0, 0.0, 0.0]
        for r in range(a, b):
            for c in range(3):
                s[c] = s[c] + float(rad[r, c])
        want = np.array(s) / (b - a)
        assert np.array_equal(got[g], want), g
    assert api.group_means(np.zeros((0, 3), np.float32), [0]).shape == (0, 3)
    for bad in ([1, n], [0, n - 1], [0, 5, 3, n]):
        with pytest.raises(ValueError):
            api.group_means(rad, bad)


PIN_SCENES = ["spheres.json", "cornell_box.json", "dupin.json", "detached_materials.json", "light_source.json",
              "torus.json"]


def _camera_groups(sc, n_pixels, spp, seed, w=64, h=48):
    """the frame's primary rays of n_pixels pixels spread over a w x h image, spp samples each, with their keys"""
    cam = sc.camera()
    pix = np.linspace(0, w * h - 1, n_pixels).astype(np.uint32)
    rays, keys = [], []
    for p in pix:
        for s in range(spp):
            u, v = po.philox_stream(seed, int(p), s, 0, 2)
            rays.append(po.get_ray(cam, w, h, int(p) % w + u, int(p) // w + v))
            keys.append((p, s))
    offsets = np.arange(0, n_pixels * spp + 1, spp, dtype=np.uint64)
    return np.array(rays), np.array(keys, np.uint32), offsets, pix


@pytest.mark.parametrize("name", PIN_SCENES)
def test_oracle_scatter_composes_into_ray_color(name):
    sc = rt.Scene.from_file(scene_path(name), random_spheres_seed=1)
    osc = po.OracleScene(sc.desc())
    for seed in (0, 2**64 - 1):
        rays, keys, offsets, pix = _camera_groups(sc, 48, 4, seed)
        for depth in (0, 1, 8):
            want = osc.group_sample_colors(rays, offsets, pix, depth, seed, threads=1)
            got = scatter_oracle.fold_paths(osc, rays, keys, depth, seed)
            assert np.array_equal(got.view(np.uint64), want.view(np.uint64)), (name, seed, depth)


def test_oracle_scatter_outputs():
    """the oracle's outputs follow the contract: zeros where an output does not apply, unit scattered directions from
    the hit point, and t / index equal to its nearest hit"""
    sc = rt.Scene.from_file(scene_path("light_source.json"), random_spheres_seed=1)
    osc = po.OracleScene(sc.desc())
    rays, keys, _, _ = _camera_groups(sc, 64, 4, 3)
    out = scatter_oracle.scatter_batch(osc, rays, keys, 0, 3)
    hit = osc.intersect_batch(rays)
    assert np.array_equal(out["index"], hit["index"])
    assert np.array_equal(out["t"], np.where(hit["index"] >= 0, hit["t"], 0.0))
    oc = out["outcome"]
    assert set(np.unique(oc).tolist()) <= {0, 1, 2} and (oc == 0).any() and (oc == 1).any()
    assert (out["index"][oc == 0] == -1).all() and (out["index"][oc != 0] >= 0).all()
    assert (out["scattered"][oc != 1] == 0).all()
    s = oc == 1
    assert np.array_equal(out["scattered"][s, :3], hit["point"][s])
    assert np.allclose(np.linalg.norm(out["scattered"][s, 3:], axis=1), 1.0, rtol=0, atol=1e-15)


def test_primary_rays_are_the_frames():
    """api.primary_rays against the oracle's ray caster and Philox stream (test_gpu_trace_group's _primary_rays, which
    reproduces the frame bit for bit)"""
    sc = rt.Scene.from_file(scene_path("cornell_box.json"), random_spheres_seed=1)
    cam = sc.camera()
    w, h, spp = 13, 7, 3
    pixels = [0, 5, 40, w * h - 1]
    for seed in (0, 1234, 2**64 - 1):
        rays, keys = api.primary_rays(cam, w, h, pixels, spp, seed)
        assert keys.dtype == np.uint32 and keys.shape == (len(pixels) * spp, 2) and keys.flags["C_CONTIGUOUS"]
        for k, (p, s) in enumerate(keys.tolist()):
            assert (p, s) == (pixels[k // spp], k % spp)
            u, v = po.philox_stream(seed, p, s, 0, 2)
            want = po.get_ray(cam, w, h, p % w + u, p // w + v)
            assert np.array_equal(rays[k].view(np.uint64), want.view(np.uint64)), (seed, p, s)
