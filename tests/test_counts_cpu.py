"""Counts frames (rt_render_start_counts) without a CUDA device: the core has no CPU fallback, so the call fails loudly;
argument checks need no device."""
import ctypes as C

import numpy as np
import pytest

import rs_pathtracing_b200 as rt
from rs_pathtracing_b200 import _ffi, api

from conftest import scene_path


def test_render_counts_fails_loudly_without_gpu():
    if rt.device_count() > 0:
        pytest.skip("GPU present")
    sc = rt.Scene.from_file(scene_path("cube_test.json"), add_random_spheres=False)
    with pytest.raises(rt.RtError, match="no CUDA device"):
        rt.GpuRenderer(sc, 12, 8).render_counts(sc.camera(), np.full((24, 32), 4, np.uint32))


def test_null_scene_or_map_is_invalid():
    cam, p = _ffi.Camera(), api.render_params(8, 8, 4, 8)
    counts = np.full(64, 4, np.uint32)
    lib = _ffi.core()
    assert lib.rt_render_start_counts(None, C.byref(cam), C.byref(p), counts.ctypes.data_as(C.c_void_p)) == _ffi.RT_ERR_INVALID
    assert lib.rt_render_start_counts(None, C.byref(cam), C.byref(p), None) == _ffi.RT_ERR_INVALID


def test_map_shape_and_dtype_are_checked():
    p = api.render_params(8, 6, 4, 8)
    for bad in (np.zeros((6, 8), np.int32), np.zeros((8, 6), np.uint32), np.zeros(48, np.uint32), [[0] * 8] * 6):
        with pytest.raises(ValueError):
            api.render_start_counts(None, _ffi.Camera(), p, bad)
