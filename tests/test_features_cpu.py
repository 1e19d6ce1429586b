"""First-hit feature buffers (rt_render_start_features) without a CUDA device: the core has no CPU fallback, so the
calls fail loudly; argument checks and the numpy restatement of the feature arithmetic need no device."""
import ctypes as C

import numpy as np
import pytest

import rs_pathtracing_b200 as rt
from rs_pathtracing_b200 import _ffi, api

from conftest import scene_path


def test_render_features_fails_loudly_without_gpu():
    if rt.device_count() > 0:
        pytest.skip("GPU present")
    sc = rt.Scene.from_file(scene_path("cube_test.json"), add_random_spheres=False)
    with pytest.raises(rt.RtError, match="no CUDA device"):
        rt.GpuRenderer(sc, 12, 8).render_features(sc.camera(), 32, 24, 4)
    with pytest.raises(rt.RtError, match="no CUDA device"):
        api.render_features(sc.device_scene(0), shape=(24, 32))


def test_null_arguments_and_frame_parameters_are_invalid_in_order():
    """the header's order: NULL scene / camera / params, then what rt_render_start rejects, then the size of the sums;
    all of it before the scene is looked at (a NULL scene with bad parameters reports the NULL)"""
    cam, p = _ffi.Camera(), api.render_params(8, 8, 4, 8)
    lib = _ffi.core()
    start = lib.rt_render_start_features
    assert start(None, C.byref(cam), C.byref(p)) == _ffi.RT_ERR_INVALID
    assert start(None, None, C.byref(p)) == _ffi.RT_ERR_INVALID
    assert start(None, C.byref(cam), None) == _ffi.RT_ERR_INVALID
    bad = api.render_params(0, 8, 4, 8)
    assert _message(lambda: start(None, C.byref(cam), C.byref(bad))) == (_ffi.RT_ERR_INVALID, "null argument")
    planes = _ffi.FeaturePlanes()
    ptr, n = C.c_void_p(), C.c_uint64()
    assert lib.rt_render_features(None, C.byref(planes), C.byref(planes)) == _ffi.RT_ERR_INVALID
    assert lib.rt_render_device_features(None, C.byref(ptr), C.byref(n)) == _ffi.RT_ERR_INVALID
    sums = (C.c_void_p * 1)(None)
    assert lib.rt_assemble_features(None, C.byref(p), sums, C.byref(planes), None) == _ffi.RT_ERR_INVALID


def _message(rc_call):
    rc = rc_call()
    return rc, _ffi.core().rt_last_error().decode()


@pytest.mark.parametrize("edit,needle", [
    (dict(width=0), "empty image"),
    (dict(samples_number=0), "zero samples"),
    (dict(max_depth=63), "max_depth"),
    (dict(shard_count=2, shard_index=2), "shard_index"),
    (dict(shard_count=17), "16 shards"),
    (dict(width=1 << 16, height=1 << 16), "image too large"),
    (dict(shard_count=2, tile_width=1 << 16, tile_height=1 << 16), "tile_width"),
    (dict(samples_number=0xFFFFFFF1), "samples_number too large"),
    # a 1-pixel-wide image with wide one-row tiles pads every shard to more than 2^64 / 72 owned pixels
    (dict(width=1, height=0xFFFFFFFF, shard_count=2, tile_width=0xFFFFFFFF, tile_height=1), "overflow"),
])
def test_rejected_parameters_name_their_reason(edit, needle):
    """every parameter rt_render_start rejects, and feature sums whose size overflows 64 bits, fail with RT_ERR_INVALID
    before any device work -- the handle is never read -- with a message naming the parameter"""
    sc = rt.Scene.from_file(scene_path("cube_test.json"), add_random_spheres=False)
    p = api.render_params(8, 8, 4, 8)
    for k, v in edit.items():
        if k in ("width", "height"):
            setattr(p.image, k, v)
        else:
            setattr(p, k, v)
    h = C.c_void_p(1)   # never dereferenced: the checks come first
    rc, msg = _message(lambda: _ffi.core().rt_render_start_features(h, C.byref(sc.camera()), C.byref(p)))
    assert rc == _ffi.RT_ERR_INVALID and needle in msg, (rc, msg)


def test_assemble_features_checks_its_arguments():
    lib = _ffi.core()
    planes = _ffi.FeaturePlanes()
    sums = (C.c_void_p * 1)(None)
    h = C.c_void_p(1)   # never dereferenced: the checks come first
    for edit, needle in ((dict(samples_number=0), "zero samples"), (dict(shard_count=17), "16 shards"),
                         (dict(width=0), "empty"), (dict(width=1 << 16, height=1 << 16), "too large")):
        p = api.render_params(8, 8, 4, 8)
        for k, v in edit.items():
            setattr(p.image if k in ("width", "height") else p, k, v)
        rc, msg = _message(lambda: lib.rt_assemble_features(h, C.byref(p), sums, C.byref(planes), None))
        assert rc == _ffi.RT_ERR_INVALID and needle in msg, (edit, msg)
    p = api.render_params(8, 8, 4, 8)
    assert lib.rt_assemble_features(h, C.byref(p), None, C.byref(planes), None) == _ffi.RT_ERR_INVALID
    assert lib.rt_assemble_features(h, C.byref(p), sums, None, None) == _ffi.RT_ERR_INVALID
    with pytest.raises(ValueError):
        api.assemble_features(None, p, [0], {"colour": 1})


def test_feature_sums_layout():
    assert api.FEATURE_SUMS_DTYPE.itemsize == 72
    assert C.sizeof(_ffi.FeaturePlanes) == 40
    assert [f[0] for f in _ffi.FeaturePlanes._fields_] == list(api.FEATURE_NAMES)


def _features_loop(index, t, normal, color, offsets):
    """the contract, one pixel and one sample at a time"""
    G = len(offsets) - 1
    out = {"albedo": np.zeros((G, 3)), "normal": np.zeros((G, 3)), "depth": np.zeros(G), "coverage": np.zeros(G),
           "shape": np.full(G, -1, np.int32)}
    for g in range(G):
        a, b = int(offsets[g]), int(offsets[g + 1])
        sa, sn, sd, hits = [0.0] * 3, [0.0] * 3, 0.0, 0
        for r in range(a, b):
            sa = [sa[c] + float(color[r, c]) for c in range(3)]
            if index[r] >= 0:
                sn = [sn[c] + float(normal[r, c]) for c in range(3)]
                sd += float(t[r])
                hits += 1
        n = np.float64(b - a)
        with np.errstate(invalid="ignore", divide="ignore"):
            out["albedo"][g] = np.array(sa) / n
            out["normal"][g] = np.array(sn) / n
            out["coverage"][g] = np.float64(hits) / n
        out["depth"][g] = sd / hits if hits else np.inf
        if b > a:
            out["shape"][g] = index[a]
    return out


def _synthetic(seed=5):
    rng = np.random.default_rng(seed)
    counts = np.array([3, 0, 1, 7, 2, 5, 0, 4, 3])
    offsets = np.concatenate([[0], np.cumsum(counts)])
    n = int(offsets[-1])
    index = rng.integers(-1, 9, n).astype(np.int32)
    index[offsets[-2]:offsets[-1]] = -1   # the last pixel: every sample misses
    t = rng.random(n) * rng.choice([1e-3, 1.0, 1e5], n)
    normal = rng.normal(size=(n, 3))
    normal /= np.linalg.norm(normal, axis=1)[:, None]
    normal[index < 0] = 0.0
    color = rng.random((n, 3))
    # signed zeros: a pixel whose only hit has a -0.0 normal component, and -0.0 colours
    index[offsets[2]] = 4
    normal[offsets[2]] = [-0.0, 1.0, -0.0]
    color[offsets[2]] = [-0.0, 0.5, -0.0]
    return index, t, normal, color, offsets, counts


def test_feature_means_against_a_loop():
    index, t, normal, color, offsets, counts = _synthetic()
    got = api.feature_means(index, t, normal, color, offsets)
    want = _features_loop(index, t, normal, color, offsets)
    for k in api.FEATURE_NAMES:
        assert got[k].dtype == want[k].dtype and got[k].shape == want[k].shape, k
        assert np.ascontiguousarray(got[k]).tobytes() == np.ascontiguousarray(want[k]).tobytes(), k
    # all-miss pixel: depth +inf, coverage 0, shape -1, normal +0.0, albedo the mean of the sky colours
    last = len(counts) - 1
    assert np.isposinf(got["depth"][last]) and got["coverage"][last] == 0.0 and got["shape"][last] == -1
    assert got["normal"][last].tobytes() == np.zeros(3).tobytes()
    # empty groups: NaN means, +inf depth, shape -1
    empty = counts == 0
    assert np.isnan(got["albedo"][empty]).all() and np.isnan(got["coverage"][empty]).all()
    assert np.isposinf(got["depth"][empty]).all() and (got["shape"][empty] == -1).all()
    # sums start at +0.0: a single -0.0 sample gives +0.0, never -0.0
    one = 2
    assert counts[one] == 1
    assert not np.signbit(got["normal"][one]).any() and not np.signbit(got["albedo"][one]).any()
    # a miss's normal contributes nothing, whatever the caller passed for it
    normal2 = normal.copy()
    normal2[index < 0] = 7.0
    again = api.feature_means(index, t, normal2, color, offsets)
    assert again["normal"].tobytes() == got["normal"].tobytes()
    # t of a miss is ignored too
    t2 = t.copy()
    t2[index < 0] = np.nan
    assert api.feature_means(index, t2, normal, color, offsets)["depth"].tobytes() == got["depth"].tobytes()


def test_feature_means_of_one_sample_per_pixel_is_the_hit_itself():
    index, t, normal, color, _, _ = _synthetic(9)
    n = len(index)
    got = api.feature_means(index, t, normal, color, np.arange(n + 1))
    hit = index >= 0
    assert got["albedo"].tobytes() == (color + 0.0).tobytes()
    assert np.array_equal(got["depth"][hit], t[hit]) and np.isposinf(got["depth"][~hit]).all()
    assert np.array_equal(got["shape"], index) and np.array_equal(got["coverage"], hit.astype(np.float64))


def test_feature_means_checks_its_inputs():
    idx, t, nrm, col, off = np.zeros(4, np.int32), np.zeros(4), np.zeros((4, 3)), np.zeros((4, 3)), [0, 2, 4]
    with pytest.raises(ValueError):
        api.feature_means(idx.astype(np.float64), t, nrm, col, off)   # integer shape indices
    with pytest.raises(ValueError):
        api.feature_means(idx, t[:3], nrm, col, off)                  # one t per ray
    with pytest.raises(ValueError):
        api.feature_means(idx, t, nrm[:, :2], col, off)
    with pytest.raises(ValueError):
        api.feature_means(idx, t, nrm, col[:3], off)
    with pytest.raises(ValueError):
        api.feature_means(idx, t, nrm, col, [0, 2, 3])                # offsets must end at len(index)
    with pytest.raises(ValueError):
        api.feature_means(idx, t, nrm, col, [1, 2, 4])                # ... and start at 0
    with pytest.raises(ValueError):
        api.feature_means(idx, t, nrm, col, [0, 3, 2, 4])             # ... and rise
