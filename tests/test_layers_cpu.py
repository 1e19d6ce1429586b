"""Bounce layers (rt_render_start_layers) without a CUDA device: the core has no CPU fallback, so the calls fail loudly;
argument checks and the numpy restatements of the layer arithmetic need no device."""
import ctypes as C

import numpy as np
import pytest

import rs_pathtracing_b200 as rt
from rs_pathtracing_b200 import _ffi, api

from conftest import scene_path


def test_render_layers_fails_loudly_without_gpu():
    if rt.device_count() > 0:
        pytest.skip("GPU present")
    sc = rt.Scene.from_file(scene_path("cube_test.json"), add_random_spheres=False)
    with pytest.raises(rt.RtError, match="no CUDA device"):
        rt.GpuRenderer(sc, 12, 8).render_layers(sc.camera(), 32, 24, 4, 3)
    with pytest.raises(rt.RtError, match="no CUDA device"):
        api.render_layers(sc.device_scene(0))


def test_null_arguments_and_layer_counts_are_invalid_in_order():
    """the header's order: NULL scene / camera / params, then n_layers outside [1, 63], then the frame parameters"""
    cam, p = _ffi.Camera(), api.render_params(8, 8, 4, 8)
    lib = _ffi.core()
    start = lambda *a: lib.rt_render_start_layers(*a)
    assert start(None, C.byref(cam), C.byref(p), 3) == _ffi.RT_ERR_INVALID
    assert start(None, None, C.byref(p), 3) == _ffi.RT_ERR_INVALID
    assert start(None, C.byref(cam), None, 3) == _ffi.RT_ERR_INVALID
    for n in (0, 64, 1000, 0xFFFFFFFF):
        assert start(None, C.byref(cam), C.byref(p), n) == _ffi.RT_ERR_INVALID
    ptr, n = C.c_void_p(), C.c_uint64()
    assert lib.rt_render_layers(None, None, C.byref(ptr), C.byref(n)) == _ffi.RT_ERR_INVALID
    assert lib.rt_render_device_layers(None, C.byref(ptr), C.byref(n)) == _ffi.RT_ERR_INVALID
    accs = (C.c_void_p * 1)(None)
    assert lib.rt_assemble_layers(None, C.byref(p), 3, accs, accs, None, None) == _ffi.RT_ERR_INVALID


def test_n_layers_is_checked_in_python():
    p = api.render_params(8, 6, 4, 8)
    for bad in (0, 64, -1, 2.0, "3", None, True):
        with pytest.raises(ValueError):
            api.render_start_layers(None, _ffi.Camera(), p, bad)
    assert api.check_n_layers(np.uint8(63)) == 63 and api.check_n_layers(1) == 1


def _layers_loop(radiance, levels, offsets, n_layers):
    """the contract, one pixel and one sample at a time"""
    out = np.zeros((n_layers, len(offsets) - 1, 3))
    for g in range(len(offsets) - 1):
        a, b = int(offsets[g]), int(offsets[g + 1])
        for layer in range(n_layers):
            s = [0.0, 0.0, 0.0]
            for r in range(a, b):
                if min(int(levels[r]), n_layers - 1) == layer:
                    s = [s[c] + float(np.float32(radiance[r, c])) for c in range(3)]
            with np.errstate(invalid="ignore", divide="ignore"):
                out[layer, g] = np.array(s) / np.float64(b - a)
    return out


def test_layer_means_against_a_loop():
    rng = np.random.default_rng(5)
    counts = np.array([3, 0, 1, 7, 2, 5, 0, 4])
    offsets = np.concatenate([[0], np.cumsum(counts)])
    n = int(offsets[-1])
    radiance = (rng.random((n, 3)) * rng.choice([1e-6, 1.0, 1e6], (n, 3))).astype(np.float32)
    radiance[0] = -0.0
    levels = rng.integers(0, 63, n)
    levels[:4] = [0, 62, 5, 5]
    for n_layers in (1, 2, 3, 9, 63):
        got = api.layer_means(radiance, levels, offsets, n_layers)
        want = _layers_loop(radiance, levels, offsets, n_layers)
        assert got.shape == (n_layers, len(counts), 3)
        assert np.array_equal(got, want, equal_nan=True), n_layers
        assert not np.signbit(got[:, 0]).any()   # sums start at +0.0
        assert np.isnan(got[:, counts == 0]).all()
    # one layer is group_means; the layers add up to it within f64 reassociation
    assert np.array_equal(api.layer_means(radiance, levels, offsets, 1)[0], api.group_means(radiance, offsets),
                          equal_nan=True)
    full = api.layer_means(radiance, levels, offsets, 63)
    ok = counts > 0
    assert np.allclose(full.sum(0)[ok], api.group_means(radiance, offsets)[ok], rtol=1e-14, atol=0)


def test_layer_means_checks_its_inputs():
    r, off = np.zeros((4, 3), np.float32), [0, 2, 4]
    with pytest.raises(ValueError):
        api.layer_means(r, [0, 1, 2], off, 2)            # one level per ray
    with pytest.raises(ValueError):
        api.layer_means(r, [0, 1, 2, 63], off, 2)        # levels 0 .. 62
    with pytest.raises(ValueError):
        api.layer_means(r, [0, 1, 2, -1], off, 2)
    with pytest.raises(ValueError):
        api.layer_means(r, [0.0, 1.0, 2.0, 3.0], off, 2)
    with pytest.raises(ValueError):
        api.layer_means(r, [0, 1, 2, 3], [0, 2, 3], 2)   # offsets must end at len(radiance)
    with pytest.raises(ValueError):
        api.layer_means(r, [0, 1, 2, 3], off, 0)


def test_path_levels_of_a_synthetic_record():
    """the last level whose record lists a path"""
    record = [{"ray": np.arange(6)}, {"ray": np.array([1, 2, 4])}, {"ray": np.array([2, 4])}, {"ray": np.array([4])}]
    got = api.path_levels(record, 6)
    assert got.dtype == np.int32
    assert got.tolist() == [0, 1, 2, 0, 3, 0]
    assert api.path_levels([], 3).tolist() == [-1, -1, -1]
