"""Committed golden fixtures (tests/golden/, written by tools/make_golden.py).

  reference_kat.json   the reference's own asserting tests for this path, as data  -> pin the oracle
                       AND the host mirror (CPU)
  intersect_*.npz      seeded ray batches + the oracle's nearest hit               -> oracle must still
                       reproduce them bit for bit (CPU); the CUDA path must too (GPU, through the C ABI)
  render_*.npz         small Philox frames of the oracle                           -> same (CPU); the CUDA
                       frame within one float ulp per path of the oracle's samples (GPU, check_frame)

The reference holds no golden vector for nearest hit / t / normal / colour (SURVEY.md 8c: "parity
unpinned"), so the npz fixtures are oracle-generated; they freeze the restatement."""
import glob
import json
import math
import os

import numpy as np
import pytest

import rs_pathtracing_b200 as rt
from oracle import pyoracle as po

from conftest import ROOT, scene_path

GOLDEN = os.path.join(ROOT, "tests", "golden")
INTERSECT = sorted(os.path.basename(p)[len("intersect_"):-4] for p in glob.glob(os.path.join(GOLDEN, "intersect_*.npz")))
RENDER = sorted(os.path.basename(p)[len("render_"):-4] for p in glob.glob(os.path.join(GOLDEN, "render_*.npz")))


def _scene(tag):
    if tag == "trio":
        from test_gpu_intersect import TRIO
        return rt.Scene.from_json(json.dumps(TRIO), add_random_spheres=False)
    return rt.Scene.from_file(scene_path(tag + ".json"), random_spheres_seed=1)


def _same(a, b):
    return ((a == b) | (np.isnan(a) & np.isnan(b))).all()


def test_fixture_inventory():
    assert {"trio", "spheres", "cornell_box", "detached_materials", "dupin"} <= set(INTERSECT)
    assert {"spheres", "cornell_box"} <= set(RENDER)


def test_reference_kat_pins_oracle_and_host_mirror():
    kat = json.load(open(os.path.join(GOLDEN, "reference_kat.json")))
    k = kat["rotate_matrix"]
    v = po.transform_point(po.mat_rotate(k["rotate_deg"]), k["point"])
    assert all(abs(a - b) < k["tol"] for a, b in zip(v, k["expected"]))
    k = kat["matrix_multiplication"]
    m1, m2 = np.array(k["m1"], dtype=float).reshape(4, 4), np.array(k["m2"], dtype=float).reshape(4, 4)
    for prod, want in ((po.mat_mul(m1, m2), k["m1m2"]), (po.mat_mul(m2, m1), k["m2m1"])):
        for key, val in want.items():
            r, c = map(int, key.split(","))
            assert prod[r][c] == val
    k = kat["bound_transform"]
    direct, _ = po.transform_new(k["translate"], k["rotate"], k["scale"])
    mn, mx = po.aabb_transform(k["aabb"][0], k["aabb"][1], direct)
    for got, want in zip(list(mn) + list(mx), k["expected"][0] + k["expected"][1]):
        assert abs(got - want) < k["tol"]
    k = kat["camera"]
    for new in (po.camera_new, rt.camera_new):   # oracle and host mirror
        cam = new(k["position"], k["direction"], k["up"], k["focal_length"], math.radians(k["fov_deg"]))
        right = (cam.right.x, cam.right.y, cam.right.z)
        assert all(abs(a - b) < k["tol"] for a, b in zip(right, k["expected_right"]))
    cam = po.camera_new(k["position"], k["direction"], k["up"], k["focal_length"], math.radians(k["fov_deg"]))
    assert abs(po.pixel_resolution(cam, *k["image"]) - k["expected_pixel_resolution"]) < k["tol"]


@pytest.mark.parametrize("tag", INTERSECT)
def test_oracle_reproduces_golden_intersections(tag):
    g = np.load(os.path.join(GOLDEN, f"intersect_{tag}.npz"))
    sc = _scene(tag)
    assert sc.shape_count == int(g["n_shapes"])
    got = po.OracleScene(sc.desc()).intersect_batch(g["rays"])
    assert np.array_equal(got["index"], g["index"])
    hit = g["index"] >= 0
    for key in ("t", "normal", "point", "uv"):
        assert _same(got[key][hit], g[key][hit]), key
    assert np.array_equal(got["front"][hit], g["front"][hit])


@pytest.mark.parametrize("tag", RENDER)
def test_oracle_reproduces_golden_frames(tag):
    g = np.load(os.path.join(GOLDEN, f"render_{tag}.npz"))
    w, h, spp, depth, seed = (int(v) for v in g["params"])
    sc = _scene(tag)
    frame, _ = po.OracleScene(sc.desc()).render(sc.camera(), w, h, spp, depth, seed=seed, rng="philox")
    assert _same(frame, g["frame"])


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [rt.RT_ISECT_BRUTE, rt.RT_ISECT_FAST])
@pytest.mark.parametrize("tag", INTERSECT)
def test_cuda_reproduces_golden_intersections(tag, mode):
    g = np.load(os.path.join(GOLDEN, f"intersect_{tag}.npz"))
    sc = _scene(tag)
    got = sc.closest_hit(g["rays"], mode=mode)
    assert np.array_equal(got["index"], g["index"])          # bit-exact nearest-hit shape index
    hit = g["index"] >= 0
    for key in ("t", "normal", "point"):                      # contract: 1e-5 relative; we require 0 ulp
        assert _same(got[key][hit], g[key][hit]), key
    assert np.allclose(got["uv"][hit], g["uv"][hit], rtol=0, atol=1e-12, equal_nan=True)
    assert np.array_equal(got["front"][hit], g["front"][hit])


@pytest.mark.gpu
@pytest.mark.parametrize("tag", RENDER)
def test_cuda_reproduces_golden_frames(tag):
    g = np.load(os.path.join(GOLDEN, f"render_{tag}.npz"))
    w, h, spp, depth, seed = (int(v) for v in g["params"])
    sc = _scene(tag)
    got = rt.GpuRenderer(sc, 12, depth, seed=seed).render(sc.camera(), w, h, spp)
    # the oracle's per-sample colours at the golden parameters (test_oracle_reproduces_golden_frames ties the oracle to
    # the file): one float ulp per path, no pixel exempt
    from test_gpu_frame_edges import check_frame
    check_frame(got, po.OracleScene(sc.desc()), sc.camera(), w, h, spp, depth, seed, f"golden {tag}")
