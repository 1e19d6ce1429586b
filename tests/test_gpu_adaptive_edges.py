"""Adaptive frames (rt_render_start_adaptive) at the edges of schedule, image, depth, seed, batching and buffer reuse.

Every case asserts the three things an adaptive frame promises (check_adaptive):
  * every pixel equals the rt_render_start frame at its own sample count, bit for bit;
  * the counts are what the documented stopping rule gives, replayed in numpy (_replay) on the moments that uniform
    frames give at each level;
  * the moments of pass 0 are within check_moments' bound of the oracle's per-sample colours (one float ulp per path).
The refinement kernels (k_adaptive_select, k_raygen_list, k_resolve_list) run in every case but depth 0, where every
sample is black and every pixel stops after pass 0 through se = 0 <= 0."""
import json

import numpy as np
import pytest

import rs_pathtracing_b200 as rt
from rs_pathtracing_b200 import api
from oracle import pyoracle as po

from conftest import scene_path
from test_gpu_adaptive import _levels, _replay, check_moments
from test_gpu_frame_edges import CAVE

pytestmark = pytest.mark.gpu


def _adaptive(hd, cam, w, h, spp, mn, rel, abs_error, depth, seed):
    api.render_start_adaptive(hd, cam, api.render_params(w, h, spp, depth, seed), mn, rel, abs_error)
    frame = np.zeros((h, w, 3))
    api.render_wait(hd, frame)
    counts, moments = api.render_pixel_stats(hd)
    return frame, counts, moments


def _uniform(hd, cam, w, h, spp, depth, seed):
    api.render_start(hd, cam, api.render_params(w, h, spp, depth, seed))
    frame = np.zeros((h, w, 3))
    api.render_wait(hd, frame)
    return frame


def check_adaptive(sc, cam, w, h, spp, mn, rel, abs_error, depth, seed, n_oracle=256):
    """one adaptive frame and the three checks; returns (frame, counts, moments)"""
    hd = sc.device_scene(0)
    frame, counts, moments = _adaptive(hd, cam, w, h, spp, mn, rel, abs_error, depth, seed)
    levels = _levels(mn, spp)
    assert set(np.unique(counts).tolist()) <= set(levels), np.unique(counts)
    moments_at = {}
    for n in levels:
        sel = counts == n
        assert np.array_equal(frame[sel], _uniform(hd, cam, w, h, n, depth, seed)[sel]), n
        moments_at[n] = _adaptive(hd, cam, w, h, n, n, 0.0, 0.0, depth, seed)[2]
    assert np.array_equal(moments_at[spp][counts == spp], moments[counts == spp])
    replay = _replay(moments_at, mn, spp, rel, abs_error)
    assert np.array_equal(replay, counts), (np.unique(replay, return_counts=True), np.unique(counts, return_counts=True))
    # pass 0 against the oracle, on every pixel of a small image or a seeded sample of a large one
    pix = np.arange(w * h)
    if w * h > n_oracle:
        pix = np.sort(np.random.default_rng(seed % 997).choice(w * h, n_oracle, replace=False))
    cols = po.OracleScene(sc.desc()).frame_sample_colors(cam, w, h, mn, depth, seed, pixels=pix)
    m0 = moments_at[mn].reshape(-1, 2)
    exact = sum(check_moments(m0[p], cols[i]) for i, p in enumerate(pix))
    print(f"moments {w}x{h} ({mn}, {spp}) depth {depth}: {len(pix) - exact} of {len(pix)} pixels not bit-identical")
    return frame, counts, moments


def _load(name):
    if name == "cave":
        return rt.Scene.from_json(json.dumps(CAVE), add_random_spheres=False)
    return rt.Scene.from_file(scene_path(name), random_spheres_seed=1)


@pytest.mark.parametrize("mn,spp,rel", [(3, 10, 0.05), (2, 3, 0.05), (7, 8, 0.05), (2, 1024, 0.01)])
def test_schedules(mn, spp, rel):
    """counts that are not min_samples times a power of two (3 -> 6 -> 10), passes of one sample (2 -> 3, 7 -> 8) and
    nine refinement passes (2 -> 1024)"""
    sc = _load("spheres.json")
    w, h = 24, 16
    _, counts, _ = check_adaptive(sc, sc.camera(), w, h, spp, mn, rel, 0.0, 8, 41)
    assert (counts > mn).any() and (counts == mn).any(), np.unique(counts, return_counts=True)


@pytest.mark.parametrize("w,h", [(1, 1), (1, 45), (45, 1), (2, 70000)])
def test_image_shapes(w, h):
    """a 1x1 image, a one-column and a one-row image, and an image taller than a grid's 65535 rows"""
    sc = _load("spheres.json")
    _, counts, _ = check_adaptive(sc, sc.camera(), w, h, 8, 2, 0.05, 0.0, 4, 1 << 32)
    if w * h > 1:
        assert (counts > 2).any(), np.unique(counts, return_counts=True)


def test_depth_zero_stops_every_pixel_at_min_samples():
    """depth 0 inside the cave: every primary ray hits, every sample is black, se = 0 <= max(rel * 0, 0)"""
    sc = _load("cave")
    frame, counts, moments = check_adaptive(sc, sc.camera(), 20, 14, 16, 2, 0.0, 0.0, 0, 3)
    assert (counts == 2).all() and (frame == 0).all() and (moments == 0).all()


def test_depth_one_constant_pixels_stop():
    """depth 1 inside the cave: a wall sample is exactly black, a lamp sample is exactly its emission; pixels whose
    samples are all equal have se == 0 and stop at min_samples, the lamp's edge goes on"""
    sc = _load("cave")
    cam = sc.camera()
    w, h = 40, 30
    frame, counts, moments = check_adaptive(sc, cam, w, h, 16, 2, 0.05, 0.0, 1, 3)
    black = (frame == 0).all(axis=2)
    lamp = (frame == 4.0).all(axis=2)
    assert black.any() and lamp.any()
    assert (counts[black | lamp] == 2).all()
    assert (counts > 2).any()


def test_depth_62():
    sc = _load("cave")
    _, counts, _ = check_adaptive(sc, sc.camera(), 12, 8, 8, 2, 0.05, 0.0, 62, 5)
    assert (counts > 2).any()


def test_absolute_error_only():
    """rel_error 0: only abs_error stops a pixel"""
    sc = _load("spheres.json")
    _, counts, _ = check_adaptive(sc, sc.camera(), 24, 16, 16, 2, 0.0, 0.01, 8, 9)
    assert (counts > 2).any() and (counts < 16).any(), np.unique(counts, return_counts=True)


@pytest.mark.parametrize("seed", [0, (1 << 64) - 1])
def test_seed_words(seed):
    sc = _load("light_source.json")
    check_adaptive(sc, sc.camera(), 24, 16, 16, 2, 0.05, 0.0, 6, seed)


def test_batches_around_a_pass(monkeypatch):
    """RT_B200_BATCH_PATHS = B*m - 1, B*m and B*m + 1 for the pass 4 -> 8 (m = 4, B = 5), on 1, 2 and 3 lanes: the
    default schedule's frame, counts and moments bit for bit"""
    w, h, spp, mn, rel, depth, seed = 20, 15, 16, 2, 0.05, 8, 12
    sc = _load("spheres.json")
    cam = sc.camera()
    ref = check_adaptive(sc, cam, w, h, spp, mn, rel, 0.0, depth, seed)
    assert len(np.unique(ref[1])) >= 3
    for cap in (19, 20, 21):
        for lanes in (1, 2, 3):
            monkeypatch.setenv("RT_B200_BATCH_PATHS", str(cap))
            monkeypatch.setenv("RT_B200_LANES", str(lanes))
            alt = _load("spheres.json")   # a new device handle reads the variables
            got = _adaptive(alt.device_scene(0), cam, w, h, spp, mn, rel, 0.0, depth, seed)
            for a, b in zip(got, ref):
                assert np.array_equal(a, b), (cap, lanes)


def test_buffers_reused_across_frame_sizes():
    """one handle renders adaptive frames of 160x120, 64x48 and 160x120 again (the moments, pixel list and live counts
    are reused, larger than the second frame needs): each equals a fresh handle's frame, counts and moments"""
    sc = _load("cornell_box.json")
    cam = sc.camera()
    hd = sc.device_scene(0)
    for w, h in ((160, 120), (64, 48), (160, 120)):
        got = _adaptive(hd, cam, w, h, 16, 2, 0.05, 0.0, 8, 7)
        fresh = _load("cornell_box.json")   # the scene owns its device handle: keep it alive while the handle is used
        want = _adaptive(fresh.device_scene(0), cam, w, h, 16, 2, 0.05, 0.0, 8, 7)
        for a, b in zip(got, want):
            assert np.array_equal(a, b), (w, h)
        assert len(np.unique(got[1])) >= 3
