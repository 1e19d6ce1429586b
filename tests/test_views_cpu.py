"""Views frames (rt_render_start_views) without a CUDA device: the core has no CPU fallback, so the call fails loudly;
argument checks need no device."""
import ctypes as C

import pytest

import rs_pathtracing_b200 as rt
from rs_pathtracing_b200 import _ffi, api

from conftest import scene_path


def test_render_views_fails_loudly_without_gpu():
    if rt.device_count() > 0:
        pytest.skip("GPU present")
    sc = rt.Scene.from_file(scene_path("cube_test.json"), add_random_spheres=False)
    with pytest.raises(rt.RtError, match="no CUDA device"):
        rt.GpuRenderer(sc, 12, 8).render_views([sc.camera(), sc.camera()], 32, 24, 4)


def test_null_scene_cameras_and_zero_views_are_invalid():
    cams, p = (_ffi.Camera * 2)(), api.render_params(8, 8, 4, 8)
    lib = _ffi.core()
    assert lib.rt_render_start_views(None, cams, 2, C.byref(p)) == _ffi.RT_ERR_INVALID
    assert lib.rt_render_start_views(None, None, 2, C.byref(p)) == _ffi.RT_ERR_INVALID
    assert lib.rt_render_start_views(None, cams, 2, None) == _ffi.RT_ERR_INVALID
    assert lib.rt_render_start_views(None, cams, 0, C.byref(p)) == _ffi.RT_ERR_INVALID


def test_camera_list_is_checked():
    p = api.render_params(8, 6, 4, 8)
    for bad in ([], (), _ffi.Camera(), [_ffi.Camera(), None], [(0, 0, 0)], 3, "cameras"):
        with pytest.raises(ValueError):
            api.render_start_views(None, bad, p)


def test_stacked_params():
    p = api.render_params(40, 30, 4, 8, seed=5, shard_count=4, shard_index=2, tile=16)
    s = api.stacked_params(p, 3)
    assert (s.image.width, s.image.height) == (40, 90)
    assert (p.image.width, p.image.height) == (40, 30)
    assert (s.samples_number, s.max_depth, s.seed, s.shard_count, s.shard_index, s.tile_width, s.tile_height) == \
        (4, 8, 5, 4, 2, 16, 16)
    assert api.shard_float4_count(s, 2) == api.shard_float4_count(api.render_params(40, 90, 4, 8, 0, 4, 2, 16), 2)


def test_orbit_cameras_turn_about_the_y_axis():
    sc = rt.Scene.from_file(scene_path("cornell_box.json"), add_random_spheres=False)
    cam = sc.camera()
    cams = api.orbit_cameras(cam, 4)
    assert len(cams) == 4 and all(isinstance(c, _ffi.Camera) for c in cams)
    px, py, pz = cam.position.tuple()
    dx, dy, dz = cam.direction.tuple()
    for c, (ex, ez) in zip(cams, [(px, pz), (pz, -px), (-px, -pz), (-pz, px)]):
        assert c.position.tuple() == pytest.approx((ex, py, ez), abs=1e-9)
        assert (c.fov_rad, c.focal_length) == (cam.fov_rad, cam.focal_length)
    assert cams[2].direction.tuple() == pytest.approx((-dx, dy, -dz), abs=1e-9)
