"""Adaptive sampling without a CUDA device: the core has no CPU fallback, so the calls fail loudly; the bindings and the
host-side helpers need no device."""
import ctypes as C
import math

import numpy as np
import pytest

import rs_pathtracing_b200 as rt
from rs_pathtracing_b200 import _ffi, api

from conftest import scene_path


def test_render_adaptive_fails_loudly_without_gpu():
    if rt.device_count() > 0:
        pytest.skip("GPU present")
    sc = rt.Scene.from_file(scene_path("cube_test.json"), add_random_spheres=False)
    with pytest.raises(rt.RtError, match="no CUDA device"):
        rt.GpuRenderer(sc, 12, 8).render_adaptive(sc.camera(), 32, 24, 16, 4, 0.05)


def test_adaptive_params_layout_and_null_arguments():
    assert C.sizeof(_ffi.AdaptiveParams) == 24
    assert [f[0] for f in _ffi.AdaptiveParams._fields_] == ["min_samples", "rel_error", "abs_error"]
    cam, p, ap = _ffi.Camera(), api.render_params(8, 8, 4, 8), _ffi.AdaptiveParams(2, 0.1, 0.0)
    lib = _ffi.core()
    assert lib.rt_render_start_adaptive(None, C.byref(cam), C.byref(p), C.byref(ap)) == _ffi.RT_ERR_INVALID
    assert lib.rt_render_pixel_stats(None, None, None) == _ffi.RT_ERR_INVALID


def test_standard_error_is_the_stopping_rule_arithmetic():
    rng = np.random.default_rng(1)
    counts = rng.choice([2, 4, 8, 64], size=(5, 7)).astype(np.uint32)
    ys = [[rng.exponential(0.3, int(n)) for n in row] for row in counts]
    moments = np.array([[[y.sum(), (y * y).sum()] for y in row] for row in ys])
    se = api.standard_error(counts, moments)
    for i in range(5):
        for j in range(7):
            n = float(counts[i, j])
            sy, syy = moments[i, j]
            mean = sy / n
            var = max(0.0, (syy - sy * mean) / (n - 1.0))
            assert se[i, j] == math.sqrt(var / n)
    # a negative variance estimate (Syy < Sy * mean) is clamped to zero
    assert api.standard_error(np.array([3], np.uint32), np.array([[1.0, 0.3]]))[0] == 0.0
