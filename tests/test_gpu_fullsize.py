"""Parity at BASELINE.json's full sizes, through properties that do not depend on the size (the oracle
finishes only small cases in seconds; here it spot-checks random subsets of the full-size result):

  cfg 2  1 Mi rays: the culled kernel == the literal-loop kernel on every ray, bit for bit; RT_ISECT_VERIFY
         finds no false cull; a random subset == the oracle
  cfg 3  1024 x 1024: the frame is independent of the batch size, of the number of lanes (streams) and of
         the number of shards (the RNG is keyed by pixel / sample / event), bit for bit; random pixels ==
         the oracle's per-sample colours for the same Philox streams; 256 spp converges to the same mean
         as 16 spp
  cfg 4  detached_materials.json at 1920 x 1080, as shipped (4a) and with every material / texture kind live and the
         camera looking at the origin (4b): the same schedule / shard independence and oracle pixel probes
  cfg 5  dupin.json at 3840 x 2160: the same, with 2 / 4 / 8 interleaved-tile shards
(cfg 4 and 5 run at reduced samples per pixel -- the resolution, tiling and batching are the configuration's)
"""
import json

import numpy as np
import pytest

import rs_pathtracing_b200 as rt
from rs_pathtracing_b200 import api
from oracle import pyoracle as po

from conftest import scene_path
from test_gpu_frame_edges import check_pixels
from test_gpu_intersect import TRIO, bench_rays, scene_rays

pytestmark = pytest.mark.gpu

N_RAYS = 1 << 20


def _same(a, b):
    return ((a == b) | (np.isnan(a) & np.isnan(b))).all()


@pytest.mark.parametrize("which", ["trio", "cornell_box"])
def test_cfg2_one_million_rays(which):
    if which == "trio":
        sc = rt.Scene.from_json(json.dumps(TRIO), add_random_spheres=False)
        rays = bench_rays(N_RAYS, seed=42)
    else:
        sc = rt.Scene.from_file(scene_path("cornell_box.json"), random_spheres_seed=1)
        rays = scene_rays(sc, N_RAYS, seed=9)
    fast = sc.closest_hit(rays, mode=rt.RT_ISECT_FAST)
    brute = sc.closest_hit(rays, mode=rt.RT_ISECT_BRUTE)
    assert np.array_equal(fast["index"], brute["index"])
    hit = brute["index"] >= 0
    assert 0.2 < hit.mean() < 0.95
    for key in ("t", "normal", "point"):
        assert _same(fast[key][hit], brute[key][hit]), key
    sub = np.random.default_rng(3).choice(N_RAYS, 8192, replace=False)
    want = po.OracleScene(sc.desc()).intersect_batch(rays[sub])
    assert np.array_equal(brute["index"][sub], want["index"])
    h = want["index"] >= 0
    for key in ("t", "normal", "point"):
        assert _same(brute[key][sub][h], want[key][h]), key
    sc.reset_stats()
    sc.closest_hit(rays[: 1 << 16], mode=rt.RT_ISECT_VERIFY, want=("index",))
    st = sc.stats()
    assert st.verify_rays == 0 and st.verify_false_culls == 0


def _frame(monkeypatch, w, h, spp, seed, batch=None, lanes=None):
    if batch is not None:
        monkeypatch.setenv("RT_B200_BATCH_PATHS", str(batch))
    if lanes is not None:
        monkeypatch.setenv("RT_B200_LANES", str(lanes))
    sc = rt.Scene.from_file(scene_path("cornell_box.json"), random_spheres_seed=1)   # env is read at scene creation / start
    frame = rt.GpuRenderer(sc, 12, 8, seed=seed).render(sc.camera(), w, h, spp)
    monkeypatch.delenv("RT_B200_BATCH_PATHS", raising=False)
    monkeypatch.delenv("RT_B200_LANES", raising=False)
    return sc, frame


def test_cfg3_full_resolution_frame_is_schedule_independent(monkeypatch):
    w = h = 1024
    spp, seed = 4, 77
    sc, ref = _frame(monkeypatch, w, h, spp, seed)
    assert np.isfinite(ref).all() and ref.mean() > 0.05
    _, small_batches = _frame(monkeypatch, w, h, spp, seed, batch=1 << 19)
    assert np.array_equal(small_batches, ref)
    _, one_lane = _frame(monkeypatch, w, h, spp, seed, lanes=1)
    assert np.array_equal(one_lane, ref)
    _, three_lanes = _frame(monkeypatch, w, h, spp, seed, lanes=3, batch=1 << 20)
    assert np.array_equal(three_lanes, ref)
    # shards: the host path of a sharded render scatters the owned pixels into the caller's buffer
    cam = sc.camera()
    for shards in (2, 8):
        buf = np.full((h, w, 3), -1.0)
        for s in range(shards):
            scn = rt.Scene.from_file(scene_path("cornell_box.json"), random_spheres_seed=1)
            ds = scn.device_scene(0)
            api.render_start(ds, cam, api.render_params(w, h, spp, 8, seed, shards, s, tile=32))
            api.render_wait(ds, buf)
        assert np.array_equal(buf, ref), shards
    # random pixels of the full-size frame against the oracle's samples of the same Philox streams
    rng = np.random.default_rng(5)
    pix = rng.integers(0, w, 96) + rng.integers(0, h, 96) * w
    cols = po.OracleScene(sc.desc()).frame_sample_colors(cam, w, h, spp, 8, seed, pixels=pix)
    check_pixels(ref.reshape(-1, 3)[pix], cols, "cfg 3 probes")


def test_cfg3_convergence_of_the_full_config():
    """1024 x 1024 x 256 (the bench workload) and 16 spp estimate the same image: mean luminance within
    0.5 %, and the per-pixel difference shrinks like the 16-spp noise (no bias that grows with spp)"""
    sc = rt.Scene.from_file(scene_path("cornell_box.json"), random_spheres_seed=1)
    cam = sc.camera()
    lum = lambda f: 0.2126 * f[..., 0] + 0.7152 * f[..., 1] + 0.0722 * f[..., 2]
    full = np.clip(rt.GpuRenderer(sc, 12, 8, seed=1).render(cam, 1024, 1024, 256), 0, 4)
    a = np.clip(rt.GpuRenderer(sc, 12, 8, seed=2).render(cam, 1024, 1024, 16), 0, 4)
    b = np.clip(rt.GpuRenderer(sc, 12, 8, seed=3).render(cam, 1024, 1024, 16), 0, 4)
    assert abs(lum(full).mean() - lum(a).mean()) / lum(full).mean() < 5e-3
    noise = np.sqrt(((a - b) ** 2).mean())            # = sqrt(2) * sigma_16
    err = np.sqrt(((a - full) ** 2).mean())           # ~ sigma_16 * sqrt(1 + 1/16)
    assert err < 0.85 * noise, (err, noise)


def _cfg_scene(cfg):
    """(scene, camera) of BASELINE.json's configurations 4a / 4b / 5 (SURVEY 8d)"""
    if cfg == "5":
        sc = rt.Scene.from_file(scene_path("dupin.json"), random_spheres_seed=1)
        return sc, sc.camera()
    sc = rt.Scene.from_file(scene_path("detached_materials.json"), random_spheres_seed=1)
    cam = sc.camera()
    if cfg == "4b":
        sc.assign_material(1, "EarthMap")        # Sphere1  -> Metal + ImageTexture
        sc.assign_material(2, "Glass")           # Cushion  -> Dielectric
        sc.assign_material(5, "Lambertian01")    # a random sphere -> Lambertian + UVChecker
        sc.assign_material(6, "WhiteMirror")
        pos = np.array(cam.position.tuple())
        cam = rt.camera_new(pos, -pos, (0, 1, 0), 1.0, cam.fov_rad)
    return sc, cam


@pytest.mark.parametrize("cfg,w,h,spp,shard_counts", [("4a", 1920, 1080, 2, (2, 8)), ("4b", 1920, 1080, 2, (2, 8)),
                                                      ("5", 3840, 2160, 1, (2, 4, 8))])
def test_cfg4_cfg5_full_resolution_frames(monkeypatch, cfg, w, h, spp, shard_counts):
    """BASELINE configs[3] and configs[4] at their own resolution: schedule independence (batch size, lanes), shard
    independence (interleaved 32x32 tiles, every shard count the scaling run uses) bit for bit, and 96 random pixels
    against the oracle's per-sample colours of the same Philox streams."""
    seed, depth = 31, 8

    def frame(batch=None, lanes=None):
        if batch is not None:
            monkeypatch.setenv("RT_B200_BATCH_PATHS", str(batch))
        if lanes is not None:
            monkeypatch.setenv("RT_B200_LANES", str(lanes))
        sc, cam = _cfg_scene(cfg)
        out = rt.GpuRenderer(sc, 12, depth, seed=seed).render(cam, w, h, spp)
        monkeypatch.delenv("RT_B200_BATCH_PATHS", raising=False)
        monkeypatch.delenv("RT_B200_LANES", raising=False)
        return sc, cam, out

    sc, cam, ref = frame()
    assert np.isfinite(ref).all() and ref.mean() > 0.05
    assert np.array_equal(frame(batch=1 << 20)[2], ref)
    assert np.array_equal(frame(lanes=1)[2], ref)
    assert np.array_equal(frame(lanes=3, batch=1 << 21)[2], ref)
    for shards in shard_counts:
        buf = np.full((h, w, 3), -1.0)
        for s in range(shards):
            scn, _ = _cfg_scene(cfg)
            ds = scn.device_scene(0)
            api.render_start(ds, cam, api.render_params(w, h, spp, depth, seed, shards, s, tile=32))
            api.render_wait(ds, buf)
        assert np.array_equal(buf, ref), shards
    rng = np.random.default_rng(11)
    pix = rng.integers(0, w, 96) + rng.integers(0, h, 96) * w
    cols = po.OracleScene(sc.desc()).frame_sample_colors(cam, w, h, spp, depth, seed, pixels=pix)
    check_pixels(ref.reshape(-1, 3)[pix], cols, f"cfg {cfg} probes")
