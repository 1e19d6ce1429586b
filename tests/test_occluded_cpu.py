"""Occlusion queries (rt_occluded_batch[_device]) without a CUDA device: the core has no CPU fallback, so the query
fails loudly; the argument checks and api.shadow_rays need no device."""
import ctypes as C
import math

import numpy as np
import pytest

import rs_pathtracing_b200 as rt
from rs_pathtracing_b200 import _ffi, api

from conftest import scene_path


@pytest.mark.skipif(rt.device_count() > 0, reason="checks the behaviour without a CUDA device")
def test_occluded_fails_loudly_without_gpu():
    sc = rt.Scene.from_file(scene_path("cube_test.json"), add_random_spheres=False)
    with pytest.raises(rt.RtError, match="no CUDA device"):
        sc.occluded(np.zeros((1, 6)))
    with pytest.raises(rt.RtError, match="no CUDA device"):
        sc.occluded(np.zeros((3, 6)), max_t=np.ones(3))
    # the device form needs a handle, and no handle can exist without a device
    out = C.c_void_p()
    assert _ffi.core().rt_scene_create(C.byref(sc.desc()), 0, C.byref(out)) == _ffi.RT_ERR_NO_DEVICE


def test_null_scene_rays_output_and_unknown_mode_are_invalid():
    lib = _ffi.core()
    rays = np.zeros((4, 6))
    occ = np.zeros(4, np.uint8)
    tmax = np.ones(4)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    for fn, extra in ((lib.rt_occluded_batch, ()), (lib.rt_occluded_batch_device, (None,))):
        assert fn(None, p(rays), 4, 0.001, math.inf, None, rt.RT_ISECT_FAST, p(occ), *extra) == _ffi.RT_ERR_INVALID
        assert fn(None, p(rays), 4, 0.001, math.inf, p(tmax), rt.RT_ISECT_BRUTE, p(occ), *extra) == _ffi.RT_ERR_INVALID
        assert fn(None, None, 4, 0.001, math.inf, None, rt.RT_ISECT_FAST, p(occ), *extra) == _ffi.RT_ERR_INVALID
        assert fn(None, p(rays), 4, 0.001, math.inf, None, rt.RT_ISECT_FAST, None, *extra) == _ffi.RT_ERR_INVALID
        assert fn(None, p(rays), 4, 0.001, math.inf, None, 7, p(occ), *extra) == _ffi.RT_ERR_INVALID
        assert fn(None, p(rays), 0, 0.001, math.inf, None, rt.RT_ISECT_FAST, p(occ), *extra) == _ffi.RT_ERR_INVALID
        assert b"null scene" in lib.rt_last_error()


def test_t_max_is_checked_before_the_call():
    sc = rt.Scene.from_file(scene_path("cube_test.json"), add_random_spheres=False)
    rays = np.zeros((6, 6))
    for bad in (np.ones(5), np.ones(7), np.ones((6, 1)), np.ones(6, np.float32), np.ones(6, np.int64),
                np.ones(12)[::2], [1.0] * 6, "1.0"):
        with pytest.raises(ValueError):
            sc.occluded(rays, max_t=bad)
    assert api.check_t_max(2.5, 6) == (2.5, None)
    assert api.check_t_max(np.float32(0.5), 6) == (0.5, None)
    a = np.arange(6.0)
    t, per_ray = api.check_t_max(a, 6)
    assert math.isinf(t) and per_ray is a


def test_device_form_checks_its_tensors():
    torch = pytest.importorskip("torch")
    rays = torch.zeros((4, 6), dtype=torch.float64)   # a host tensor: rejected before any device work
    with pytest.raises(ValueError):
        api.occluded_device(None, rays, torch.zeros(4, dtype=torch.uint8))


def test_shadow_rays_against_numpy():
    rng = np.random.default_rng(3)
    p = rng.normal(size=(1000, 3)) * 5.0
    q = rng.normal(size=(1000, 3)) * 5.0
    rays, dist = api.shadow_rays(p, q)
    assert rays.shape == (1000, 6) and dist.shape == (1000,) and rays.flags["C_CONTIGUOUS"]
    assert np.array_equal(rays[:, :3], p)
    d = q - p
    ln = np.sqrt((d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2])
    assert np.array_equal(dist, ln)
    assert np.array_equal(rays[:, 3:], d / ln[:, None])
    assert np.allclose(dist, np.linalg.norm(d, axis=1), rtol=1e-15, atol=0)
    assert np.allclose(rays[:, :3] + rays[:, 3:] * dist[:, None], q, rtol=0, atol=1e-12)
    assert np.array_equal(api.make_rays(p, d), rays)
    with pytest.raises(ValueError):
        api.shadow_rays(p, q[:10])
