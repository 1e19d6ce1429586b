"""rt_render_start_adaptive / rt_render_pixel_stats: adaptive sampling with per-pixel sample counts.

Every pixel of an adaptive frame must equal, bit for bit, the rt_render_start frame's pixel at the count it ended with
-- i.e. trace_pixel_samples_group over its first counts[p] camera rays -- and the counts must be what the documented
stopping rule gives on the pixel's own luminance moments, whatever the batch size, the lanes or the kernel timing.
"""
import ctypes as C

import numpy as np
import pytest

import rs_pathtracing_b200 as rt
from rs_pathtracing_b200 import _ffi, api
from oracle import pyoracle as po

from conftest import scene_path

pytestmark = pytest.mark.gpu

DEPTH = 8


def _variant_4b(sc):
    """config 4b (SURVEY 8d): every material / texture kind live, camera looking at the origin"""
    sc.assign_material(1, "EarthMap")
    sc.assign_material(2, "Glass")
    sc.assign_material(5, "Lambertian01")
    sc.assign_material(6, "WhiteMirror")
    c0 = sc.camera()
    pos = np.array(c0.position.tuple())
    return rt.camera_new(pos, -pos, (0, 1, 0), 1.0, c0.fov_rad)


def _load(name, variant=""):
    sc = rt.Scene.from_file(scene_path(name), random_spheres_seed=1)
    cam = _variant_4b(sc) if variant == "4b" else sc.camera()
    return sc, cam


def _adaptive(sc, cam, w, h, spp, min_samples, rel, abs_error=0.0, seed=5):
    """(frame, counts, moments) of one adaptive frame through the raw calls"""
    ds = sc.device_scene(0)
    api.render_start_adaptive(ds, cam, api.render_params(w, h, spp, DEPTH, seed), min_samples, rel, abs_error)
    frame = np.zeros((h, w, 3))
    api.render_wait(ds, frame)
    counts, moments = api.render_pixel_stats(ds)
    return frame, counts, moments


def _uniform(sc, cam, w, h, spp, seed=5):
    ds = sc.device_scene(0)
    api.render_start(ds, cam, api.render_params(w, h, spp, DEPTH, seed))
    frame = np.zeros((h, w, 3))
    api.render_wait(ds, frame)
    return frame


def _levels(min_samples, spp):
    """the counts a pixel can hold: min * 2^j below spp, and spp"""
    out, n = [], min_samples
    while n < spp:
        out.append(n)
        n += min(n, spp - n)
    return out + [spp]


def _replay(moments_at, min_samples, spp, rel, abs_error):
    """the stopping rule of rt_b200.h in numpy, from the moments each pixel had when it was tested"""
    levels = _levels(min_samples, spp)
    counts = np.full(moments_at[levels[0]].shape[:2], levels[0], np.uint32)
    for n in levels[:-1]:
        sy, syy = moments_at[n][..., 0], moments_at[n][..., 1]
        mean = sy / n
        var = np.fmax(0.0, (syy - sy * mean) / (n - 1))
        se = np.sqrt(var / n)
        go = (counts == n) & ~(se <= np.fmax(rel * np.fabs(mean), abs_error))
        counts[go] = n + min(n, spp - n)
    return counts


def _luminance_sums(cols):
    """sequential f64 sums of y and y*y over float32-rounded sample colours"""
    c = cols.astype(np.float32).astype(np.float64)
    sy = syy = 0.0
    for r, g, b in c:
        y = (0.2126 * r + 0.7152 * g) + 0.0722 * b
        sy += y
        syy += y * y
    return sy, syy


def check_moments(got, cols):
    """got: a pixel's (sum y, sum y^2) from the device; cols: the oracle's FP64 colours of its samples, in order.  Each path
    may be one float ulp off per channel (check_pixels' rule), so with f_s the float-rounded colours and
        dy_s = 0.2126 ulp32(r_s) + 0.7152 ulp32(g_s) + 0.0722 ulp32(b_s)
    the device's sums must satisfy
        |sum y - sum y_emu| <= sum dy_s + n ulp64(sum y_emu),
        |sum y^2 - sum y^2_emu| <= sum (2 |y_s| dy_s + dy_s^2) + n ulp64(sum y^2_emu).
    Returns True when both sums are bit-identical to the emulated ones."""
    f32 = np.asarray(cols, dtype=np.float64).astype(np.float32)
    want = _luminance_sums(cols)
    sp = np.spacing(np.abs(f32)).astype(np.float64)
    dy = 0.2126 * sp[:, 0] + 0.7152 * sp[:, 1] + 0.0722 * sp[:, 2]
    f = f32.astype(np.float64)
    y = (0.2126 * f[:, 0] + 0.7152 * f[:, 1]) + 0.0722 * f[:, 2]
    n = len(f)
    b1 = dy.sum() + n * np.spacing(abs(want[0]))
    b2 = (2 * np.abs(y) * dy + dy * dy).sum() + n * np.spacing(abs(want[1]))
    got = tuple(float(v) for v in got)
    assert abs(got[0] - want[0]) <= b1 and abs(got[1] - want[1]) <= b2, (got, want, (b1, b2))
    return got == want


UNIFORM_CASES = [("spheres.json", ""), ("cornell_box.json", ""), ("detached_materials.json", "4b")]


@pytest.mark.parametrize("name,variant", UNIFORM_CASES)
def test_min_equal_to_samples_is_the_frame(name, variant):
    """min_samples == samples_number: the rt_render_start frame bit for bit, every count samples_number, and the moments
    the oracle's per-sample colours give"""
    w, h, spp, seed = 64, 48, 8, 21
    sc, cam = _load(name, variant)
    frame, counts, moments = _adaptive(sc, cam, w, h, spp, spp, 0.0, seed=seed)
    assert np.array_equal(frame, _uniform(sc, cam, w, h, spp, seed=seed))
    assert (counts == spp).all()
    # a huge rel_error stops every pixel after pass 0: the min_samples frame
    f4, c4, m4 = _adaptive(sc, cam, w, h, spp, 4, 1e300, seed=seed)
    assert (c4 == 4).all() and np.array_equal(f4, _uniform(sc, cam, w, h, 4, seed=seed))
    osc = po.OracleScene(sc.desc())
    rng = np.random.default_rng(2)
    exact = 0
    for x, y in zip(rng.integers(0, w, 24), rng.integers(0, h, 24)):
        x, y = int(x), int(y)
        cols = osc.pixel_sample_colors(cam, w, h, x, y, spp, DEPTH, seed=seed)
        same = check_moments(moments[y, x], cols)
        c32 = cols.astype(np.float32).astype(np.float64)
        rgb = np.zeros(3)
        for c in c32:
            rgb = rgb + c
        if np.array_equal(rgb / spp, frame[y, x]):
            # the oracle reproduces this pixel's float radiance exactly: its moments must match bit for bit
            assert same, (x, y, tuple(moments[y, x]), _luminance_sums(cols))
        exact += same
    print(f"moments: {24 - exact} of 24 pixels not bit-identical")
    assert exact >= 20, exact


def _camera_rays(cam, w, h, counts, seed):
    """each pixel's first counts[p] primary rays (MultisamplerRayCaster::next, Philox draws of event 0), grouped by
    pixel in x + y*w order"""
    flat = counts.reshape(-1)
    rays = np.empty((int(flat.sum()), 6))
    k = 0
    for p, n in enumerate(flat):
        x, y = p % w, p // w
        for s in range(int(n)):
            u, v = po.philox_stream(seed, p, s, 0, 2)
            rays[k] = po.get_ray(cam, w, h, x + u, y + v)
            k += 1
    offsets = np.concatenate([[0], np.cumsum(flat)]).astype(np.uint64)
    return rays, offsets


@pytest.mark.parametrize("name,variant", [("spheres.json", ""), ("cornell_box.json", ""), ("dupin.json", ""),
                                          ("detached_materials.json", "4b")])
def test_every_pixel_is_its_own_trace(name, variant):
    """160x120, min 4, at most 64 samples, rel_error 0.05: every pixel equals trace_pixel_samples_group over its first
    counts[p] camera rays and the uniform frame of counts[p] samples, bit for bit; the counts take the documented values,
    and both early stops and capped pixels occur"""
    w, h, spp, mn, rel, seed = 160, 120, 64, 4, 0.05, 7
    sc, cam = _load(name, variant)
    frame, counts, moments = _adaptive(sc, cam, w, h, spp, mn, rel, seed=seed)
    levels = _levels(mn, spp)
    assert set(np.unique(counts)) <= set(levels)
    assert (counts < spp).any() and (counts == spp).any(), np.unique(counts, return_counts=True)
    for n in levels:
        sel = counts == n
        if sel.any():
            assert np.array_equal(frame[sel], _uniform(sc, cam, w, h, n, seed=seed)[sel]), n
    rays, offsets = _camera_rays(cam, w, h, counts, seed)
    got = sc.trace_pixel_samples_group(rays, offsets, np.arange(w * h, dtype=np.uint32), DEPTH, seed=seed)
    assert np.array_equal(got, frame.reshape(-1, 3))


@pytest.mark.parametrize("name,rel,abs_error", [("spheres.json", 0.05, 0.0), ("cornell_box.json", 0.02, 1e-3)])
def test_counts_follow_the_documented_rule(name, rel, abs_error):
    """uniform frames at every level give the moments each pixel had when it was tested; the rule replayed in numpy
    reproduces the counts exactly"""
    w, h, spp, mn, seed = 96, 72, 32, 2, 3
    sc, cam = _load(name)
    _, counts, moments = _adaptive(sc, cam, w, h, spp, mn, rel, abs_error, seed=seed)
    moments_at = {n: _adaptive(sc, cam, w, h, n, n, 0.0, seed=seed)[2] for n in _levels(mn, spp)}
    assert np.array_equal(moments_at[spp][counts == spp], moments[counts == spp])
    replay = _replay(moments_at, mn, spp, rel, abs_error)
    assert np.array_equal(replay, counts), (np.unique(replay, return_counts=True), np.unique(counts, return_counts=True))
    assert len(np.unique(counts)) >= 3


def test_results_do_not_depend_on_the_schedule(monkeypatch):
    """one pixel per batch, batches of exactly RT_B200_BATCH_PATHS paths, 1 / 2 / 3 lanes, kernel timing on: frame,
    counts and moments identical bit for bit"""
    name, w, h, spp, mn, rel, seed = "spheres.json", 32, 24, 16, 2, 0.05, 11
    sc, cam = _load(name)
    ref = _adaptive(sc, cam, w, h, spp, mn, rel, seed=seed)
    assert len(np.unique(ref[1])) >= 3

    def run(env, timing=False):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        alt, _ = _load(name)   # a new device handle reads the variables
        if timing:
            alt.set_kernel_timing(True)
        got = _adaptive(alt, cam, w, h, spp, mn, rel, seed=seed)
        for k in env:
            monkeypatch.delenv(k)
        return got

    for env in ({"RT_B200_BATCH_PATHS": "1"}, {"RT_B200_BATCH_PATHS": "16"},
                {"RT_B200_BATCH_PATHS": "64", "RT_B200_LANES": "1"},
                {"RT_B200_BATCH_PATHS": "64", "RT_B200_LANES": "2"},
                {"RT_B200_BATCH_PATHS": "64", "RT_B200_LANES": "3"}):
        got = run(env)
        for a, b in zip(got, ref):
            assert np.array_equal(a, b), env
    got = run({}, timing=True)
    for a, b in zip(got, ref):
        assert np.array_equal(a, b), "kernel timing"


def _raw_start(handle, cam, params, mn, rel, abs_error=0.0):
    ap = _ffi.AdaptiveParams(mn, rel, abs_error)
    return _ffi.core().rt_render_start_adaptive(handle, C.byref(cam), C.byref(params), C.byref(ap))


def test_state_and_errors():
    w, h, spp, depth, seed = 64, 48, 16, DEPTH, 9
    sc, cam = _load("cornell_box.json")
    ds = sc.device_scene(0)
    # poll before completion: done = 0 and the buffer untouched; stop drains
    big = api.render_params(512, 512, 256, depth, seed)
    api.render_start_adaptive(ds, cam, big, 4, 0.001)
    buf = np.full((512, 512, 3), -1.0)
    assert not api.render_poll(ds, buf)
    assert (buf == -1.0).all()
    assert _ffi.core().rt_render_stop(ds) == _ffi.RT_OK
    with pytest.raises(rt.RtError, match="-4"):
        api.render_poll(ds, buf)
    # a completed frame: poll delivers it whole, the stats count every traced path, the device views work
    sc.reset_stats()
    frame, counts, moments = _adaptive(sc, cam, w, h, spp, 2, 0.05, seed=seed)
    assert sc.stats().paths == int(counts.sum())
    assert api.render_accumulated_samples(ds) == 0
    dptr, n = api.render_device_result(ds)
    assert n == w * h and dptr
    assert np.array_equal(api.tonemap_last_frame(ds).reshape(h, w, 4), rt.tonemap_rgba8(sc, frame))
    # the frame never seeds a progressive accumulation: the next accumulating frame starts afresh
    api.render_set_accumulate(ds, True)
    api.render_start_adaptive(ds, cam, api.render_params(w, h, spp, depth, seed), 2, 0.05)
    api.render_wait(ds, None)
    acc = _uniform(sc, cam, w, h, 4, seed=seed)
    assert api.render_accumulated_samples(ds) == 4
    api.render_set_accumulate(ds, False)
    assert np.array_equal(acc, _uniform(sc, cam, w, h, 4, seed=seed))
    # pixel stats of a plain frame: counts yes, moments no
    counts4, moments4 = api.render_pixel_stats(ds)
    assert (counts4 == 4).all() and moments4 is None
    m = np.empty((h, w, 2))
    assert _ffi.core().rt_render_pixel_stats(ds, None, m.ctypes.data_as(C.c_void_p)) == _ffi.RT_ERR_STATE
    # rejected parameters
    p = api.render_params(w, h, spp, depth, seed)
    for mn, rel, ab in ((1, 0.1, 0.0), (0, 0.1, 0.0), (spp + 1, 0.1, 0.0), (2, -0.1, 0.0), (2, float("nan"), 0.0),
                        (2, float("inf"), 0.0), (2, 0.1, -1.0), (2, 0.1, float("inf"))):
        assert _raw_start(ds, cam, p, mn, rel, ab) == _ffi.RT_ERR_INVALID, (mn, rel, ab)
    sharded = api.render_params(w, h, spp, depth, seed, shard_count=2, shard_index=0, tile=16)
    assert _raw_start(ds, cam, sharded, 2, 0.1) == _ffi.RT_ERR_INVALID
    assert _ffi.core().rt_render_start_adaptive(ds, C.byref(cam), C.byref(p), None) == _ffi.RT_ERR_INVALID


def test_fused_fallback_is_rejected(monkeypatch):
    monkeypatch.setenv("RT_B200_FUSED_BOUNCE", "1")
    sc, cam = _load("spheres.json")
    p = api.render_params(32, 24, 8, DEPTH, 1)
    assert _raw_start(sc.device_scene(0), cam, p, 2, 0.1) == _ffi.RT_ERR_STATE


def test_multi_device_handle_is_rejected():
    n_dev = rt.device_count()
    if n_dev < 2:
        pytest.skip("needs two GPUs")
    sc, cam = _load("spheres.json")
    h = sc.device_scene_multi(list(range(n_dev)))
    assert _raw_start(h, cam, api.render_params(32, 24, 8, DEPTH, 1), 2, 0.1) == _ffi.RT_ERR_INVALID


def test_python_renderer_returns_the_raw_results():
    w, h, spp, mn, rel, seed = 80, 60, 32, 4, 0.05, 13
    sc, cam = _load("cornell_box.json")
    frame, counts, std_error = rt.GpuRenderer(sc, 12, DEPTH, seed=seed).render_adaptive(cam, w, h, spp, mn, rel)
    other, _ = _load("cornell_box.json")
    f2, c2, m2 = _adaptive(other, cam, w, h, spp, mn, rel, seed=seed)
    assert np.array_equal(frame, f2) and np.array_equal(counts, c2)
    assert np.array_equal(std_error, api.standard_error(c2, m2))
    mean = m2[..., 0] / c2
    stopped = counts < spp
    assert (std_error[stopped] <= np.fmax(rel * np.fabs(mean[stopped]), 0.0)).all()
