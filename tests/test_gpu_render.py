"""GPU parity of the wavefront renderer against the oracle.

Two kinds of checks:
  * SAME paths: the oracle run with the shared Philox schedule follows exactly the GPU's paths, so
    EVERY pixel agrees with the oracle's samples rounded to float and summed like the GPU sums them, within one
    float ulp per path (check_pixels, tests/test_gpu_frame_edges.py); NO pixel may exceed it.
  * INDEPENDENT streams: against an oracle render with an unrelated RNG the frames must agree within
    the statistical tolerance of SURVEY §8(d): RMSE <= 1.25 * r0 + 1e-3 with r0 the oracle-vs-oracle
    noise floor, and mean luminance within 0.5 % (+ a noise allowance at the tiny test sizes).
"""
import ctypes as C
import math
import os

import numpy as np
import pytest

import rs_pathtracing_b200 as rt
from rs_pathtracing_b200 import api
from oracle import pyoracle as po

from conftest import scene_path
from test_gpu_frame_edges import check_frame

pytestmark = pytest.mark.gpu


def gpu_frame(sc, cam, w, h, spp, depth, seed):
    r = rt.GpuRenderer(sc, 12, depth, seed=seed)
    return r.render(cam, w, h, spp)


@pytest.mark.parametrize("name,w,h,spp,depth", [
    ("spheres.json", 64, 48, 4, 8),
    ("cornell_box.json", 48, 48, 4, 8),
    ("detached_materials.json", 64, 36, 4, 8),
    ("dupin.json", 64, 36, 4, 8),
    ("cube_test.json", 48, 48, 4, 50),
    ("light_source.json", 64, 36, 4, 8),     # NoiseTexture (Perlin turbulence) on the big sphere and the ground
])
def test_same_paths_as_oracle(name, w, h, spp, depth):
    sc = rt.Scene.from_file(scene_path(name), random_spheres_seed=1)
    cam = sc.camera()
    got = gpu_frame(sc, cam, w, h, spp, depth, seed=1234)
    check_frame(got, po.OracleScene(sc.desc()), cam, w, h, spp, depth, 1234, name)


def test_same_paths_all_material_and_texture_branches():
    """config 4b: look at the origin and make every material / texture kind live"""
    sc = rt.Scene.from_file(scene_path("detached_materials.json"), random_spheres_seed=1)
    sc.assign_material(1, "EarthMap")        # Sphere1  -> Metal + ImageTexture
    sc.assign_material(2, "Glass")           # Cushion  -> Dielectric
    sc.assign_material(5, "Lambertian01")    # a random sphere -> Lambertian + UVChecker
    sc.assign_material(6, "WhiteMirror")
    c0 = sc.camera()
    pos = np.array(c0.position.tuple())
    cam = rt.camera_new(pos, -pos, (0, 1, 0), 1.0, c0.fov_rad)
    w, h, spp, depth = 96, 54, 4, 8
    got = gpu_frame(sc, cam, w, h, spp, depth, seed=99)
    check_frame(got, po.OracleScene(sc.desc()), cam, w, h, spp, depth, 99, "cfg 4b")


def luminance(img):
    return 0.2126 * img[..., 0] + 0.7152 * img[..., 1] + 0.0722 * img[..., 2]


def display(img):  # main_raylib.rs:240-245 before quantisation
    return np.minimum(np.sqrt(np.maximum(img, 0)), 0.999)


def _variant_4b(sc):
    """config 4b (SURVEY 8d): every material / texture kind live, camera looking at the origin"""
    sc.assign_material(1, "EarthMap")        # Sphere1  -> Metal + ImageTexture
    sc.assign_material(2, "Glass")           # Cushion  -> Dielectric
    sc.assign_material(5, "Lambertian01")    # a random sphere -> Lambertian + UVChecker
    sc.assign_material(6, "WhiteMirror")
    c0 = sc.camera()
    pos = np.array(c0.position.tuple())
    return rt.camera_new(pos, -pos, (0, 1, 0), 1.0, c0.fov_rad)


# BASELINE.md's gate names configurations 1, 3, 4 and 5: spheres, cornell_box, detached_materials (as shipped = 4a and
# the all-branches variant 4b) and dupin
@pytest.mark.parametrize("name,variant", [("spheres.json", ""), ("cornell_box.json", ""), ("detached_materials.json", ""),
                                          ("detached_materials.json", "4b"), ("dupin.json", "")])
def test_statistical_agreement_with_independent_oracle(name, variant):
    sc = rt.Scene.from_file(scene_path(name), random_spheres_seed=1)
    cam = _variant_4b(sc) if variant == "4b" else sc.camera()
    w, h, spp, depth = 48, 36, 64, 8
    osc = po.OracleScene(sc.desc())
    a, _ = osc.render(cam, w, h, spp, depth, seed=1, rng="xoshiro", use_bvh=True)
    b, _ = osc.render(cam, w, h, spp, depth, seed=2, rng="xoshiro", use_bvh=True)
    g = gpu_frame(sc, cam, w, h, spp, depth, seed=3)
    for f in (display, lambda x: np.clip(x, 0, 4)):
        r0 = np.sqrt(((f(a) - f(b)) ** 2).mean(axis=(0, 1)))
        rg = np.sqrt(((f(g) - f(a)) ** 2).mean(axis=(0, 1)))
        assert (rg <= 1.25 * r0 + 1e-3).all(), (rg, r0)
    la, lb, lg = luminance(np.clip(a, 0, 4)).mean(), luminance(np.clip(b, 0, 4)).mean(), luminance(np.clip(g, 0, 4)).mean()
    noise = abs(la - lb) / la
    assert abs(lg - la) / la <= 0.005 + 2.0 * noise, (lg, la, lb)


def test_trace_pixel_samples_matches_oracle():
    sc = rt.Scene.from_file(scene_path("spheres.json"), random_spheres_seed=1)
    cam = sc.camera()
    osc = po.OracleScene(sc.desc())
    rng = np.random.default_rng(0)
    from test_gpu_caller_rays import check_groups
    for pix in (0, 17, 640 * 240 + 320):
        x, y = pix % 640, pix // 640
        rays = np.array([po.get_ray(cam, 640, 480, x + u, y + v) for u, v in rng.uniform(0, 1, (10, 2))])
        got = sc.trace_pixel_samples(rays, 10, seed=5, pixel_index=pix)
        cols = osc.group_sample_colors(rays, [0, 10], [pix], 10, seed=5)
        check_groups(got, cols, [0, 10], f"trace_pixel_samples pixel {pix}")


def test_renderer_trait_behaviour():
    sc = rt.Scene.from_file(scene_path("cube_test.json"), random_spheres_seed=1)
    cam = sc.camera()
    r = rt.GpuRenderer(sc, 12, 8, seed=1)
    buf = np.full((32 * 24, 3), -1.0)
    assert r.render_step(buf) is False and (buf == -1.0).all()      # nothing started: nothing written
    r.start_rendering(cam, rt.ImageParams(32, 24), 2)
    while not r.render_step(buf):
        pass
    assert (buf >= 0).all()
    first = buf.copy()
    assert r.render_step(buf) is False                               # frame consumed
    # restart overwrites, never accumulates (step_by_step.rs:115-117); same seed -> same frame
    r.start_rendering(cam, rt.ImageParams(32, 24), 2)
    while not r.render_step(buf):
        pass
    assert np.array_equal(first, buf)
    r.start_rendering(cam, rt.ImageParams(32, 24), 2)
    r.stop_rendering()
    assert r.render_step(buf) is False
    r.start_rendering(cam, rt.ImageParams(32, 24), 2)
    with pytest.raises(rt.RtError, match="shorter"):
        r.render_step(np.zeros((10, 3)))
    r.stop_rendering()


def test_progressive_delivery_and_batching(monkeypatch):
    """small batches: pixels arrive over several render_step calls, final image independent of batching"""
    sc = rt.Scene.from_file(scene_path("cube_test.json"), random_spheres_seed=1)
    cam = sc.camera()
    ref = gpu_frame(sc, cam, 64, 64, 4, 8, seed=4)
    monkeypatch.setenv("RT_B200_BATCH_PATHS", "2048")
    sc2 = rt.Scene.from_file(scene_path("cube_test.json"), random_spheres_seed=1)
    r = rt.GpuRenderer(sc2, 12, 8, seed=4)
    buf = np.full((64, 64, 3), -1.0)
    r.start_rendering(cam, rt.ImageParams(64, 64), 4)
    polls = 0
    while not r.render_step(buf):
        polls += 1
    assert np.array_equal(buf, ref)


def test_progressive_accumulation_across_start_calls():
    """rt_render_set_accumulate (SURVEY 8f-3): k frames of n samples with an unchanged camera trace the very
    paths of one frame of k*n samples -- sample indices continue where the previous frame stopped -- and deliver
    the mean over all of them; a different camera / seed / image, or toggling the switch, starts afresh"""
    w, h, depth, seed = 64, 48, 8, 9
    sc = rt.Scene.from_file(scene_path("cornell_box.json"), random_spheres_seed=1)
    cam = sc.camera()
    other = rt.Scene.from_file(scene_path("cornell_box.json"), random_spheres_seed=1)   # references: a handle of their own
    ref12 = gpu_frame(other, cam, w, h, 12, depth, seed)
    ref4 = gpu_frame(other, cam, w, h, 4, depth, seed)
    ds = sc.device_scene(0)
    api.render_set_accumulate(ds, True)
    assert api.render_accumulated_samples(ds) == 0
    buf = np.zeros((h, w, 3))
    for k in range(3):
        api.render_start(ds, cam, api.render_params(w, h, 4, depth, seed))
        api.render_wait(ds, buf)
        assert api.render_accumulated_samples(ds) == 4 * (k + 1)
        if k == 0:
            assert np.array_equal(buf, ref4)
    # the same paths, summed in the same order into f64 sums: three frames of 4 samples ARE the frame of 12
    assert np.array_equal(buf, ref12)
    assert not np.allclose(buf, ref4, rtol=1e-3, atol=1e-4)
    # device-side result carries the total sample count
    torch = pytest.importorskip("torch")
    ptr, n = api.render_device_result(ds)
    assert n == w * h
    # another seed starts afresh
    api.render_start(ds, cam, api.render_params(w, h, 4, depth, seed + 1))
    api.render_wait(ds, buf)
    assert api.render_accumulated_samples(ds) == 4
    assert np.array_equal(buf, gpu_frame(other, cam, w, h, 4, depth, seed + 1))
    # switching it off and on empties the accumulator; off = the reference's behaviour (every frame from scratch)
    api.render_set_accumulate(ds, False)
    for _ in range(2):
        api.render_start(ds, cam, api.render_params(w, h, 4, depth, seed))
        api.render_wait(ds, buf)
        assert np.array_equal(buf, ref4)
    assert api.render_accumulated_samples(ds) == 0


def test_sharded_render_assembles_to_the_unsharded_frame():
    """interleaved tiles: N shards rendered independently assemble bit-for-bit to the 1-shard frame"""
    torch = pytest.importorskip("torch")
    w, h, spp, depth, seed = 100, 70, 3, 8, 11
    sc = rt.Scene.from_file(scene_path("spheres.json"), random_spheres_seed=1)
    cam = sc.camera()
    ref = gpu_frame(sc, cam, w, h, spp, depth, seed)
    for shards in (2, 3, 8):
        scenes = [rt.Scene.from_file(scene_path("spheres.json"), random_spheres_seed=1) for _ in range(shards)]
        ptrs = []
        host_frame = np.full((h, w, 3), -1.0)
        for s, scn in enumerate(scenes):
            p = api.render_params(w, h, spp, depth, seed, shards, s, tile=32)
            ds = scn.device_scene(0)
            api.render_start(ds, cam, p)
            api.render_wait(ds, host_frame)          # host path of a sharded render scatters owned pixels
            ptr, n = api.render_device_result(ds)
            assert n == api.shard_float4_count(p, s)
            ptrs.append(ptr)
        assert np.array_equal(host_frame, ref)
        frame = torch.empty((h, w, 3), dtype=torch.float64, device="cuda")
        p0 = api.render_params(w, h, spp, depth, seed, shards, 0, tile=32)
        api.assemble_frame(scenes[0].device_scene(0), p0, ptrs, frame.data_ptr())
        torch.cuda.synchronize()
        # the accumulators hold the f64 sums themselves: the assembled frame IS the unsharded one
        assert np.array_equal(frame.cpu().numpy(), ref)


def test_one_handle_over_all_devices_renders_the_unsharded_frame():
    """rt_scene_create_multi through GpuRenderer(devices=[...]): ONE process, ONE handle, every visible GPU (all of
    them; twice the same box's device 0 is not allowed, so a single-GPU box checks the n = 1 path of the same entry
    points) -- the frame equals the single-device frame bit for bit, also with changing sizes / sample counts back to
    back, progressive accumulation and the device-side tonemap"""
    n_dev = rt.device_count()
    devices = list(range(n_dev))
    w, h, depth, seed = 200, 120, 8, 5
    sc = rt.Scene.from_file(scene_path("cornell_box.json"), random_spheres_seed=1)
    cam = sc.camera()
    multi = rt.GpuRenderer(sc, 12, depth, seed=seed, devices=devices)
    ds = sc.device_scene_multi(devices) if n_dev > 1 else sc.device_scene(0)
    assert _ffi_core().rt_scene_device_count(ds) == n_dev
    for (ww, hh, spp) in ((w, h, 4), (w, h, 2), (96, 72, 3), (w, h, 4)):
        ref_sc = rt.Scene.from_file(scene_path("cornell_box.json"), random_spheres_seed=1)
        ref = gpu_frame(ref_sc, cam, ww, hh, spp, depth, seed)
        got = multi.render(cam, ww, hh, spp)
        assert np.array_equal(got, ref), (ww, hh, spp)
        # the frame stays on the (first) device; the bins' tonemap runs on it without the f64 frame crossing the bus
        rgba = api.tonemap_last_frame(ds).reshape(hh, ww, 4)
        assert np.array_equal(rgba, rt.tonemap_rgba8(ref_sc, ref))
    # progressive accumulation through the same handle
    api.render_set_accumulate(ds, True)
    buf = np.zeros((h, w, 3))
    for k in range(3):
        api.render_start(ds, cam, api.render_params(w, h, 2, depth, seed))
        api.render_wait(ds, buf)
    api.render_set_accumulate(ds, False)
    ref_sc = rt.Scene.from_file(scene_path("cornell_box.json"), random_spheres_seed=1)
    assert np.array_equal(buf, gpu_frame(ref_sc, cam, w, h, 6, depth, seed))


def _ffi_core():
    from rs_pathtracing_b200 import _ffi
    return _ffi.core()


def test_tonemap_matches_the_bins_formula():
    sc = rt.Scene.from_file(scene_path("cube_test.json"), add_random_spheres=False)
    rng = np.random.default_rng(0)
    frame = rng.uniform(0, 2, (50, 40, 3))
    frame[0, 0] = [0.0, 4.0, math.nan]
    got = rt.tonemap_rgba8(sc, frame)
    want = (np.clip(np.sqrt(frame), 0, 0.999) * 256.0)
    want = np.where(np.isnan(want), 0, want).astype(np.uint8)
    assert np.array_equal(got[..., :3], want) and (got[..., 3] == 255).all()


def test_work_counters_match_oracle():
    """the instrumented kernels see the same segments as the oracle's brute-force loop; most (segment,
    shape) pairs are settled by the FP32 cull tree without even being looked at, the exact FP64 test runs
    on a small rest, and the number of march evaluations is much smaller (exact skipping)"""
    sc = rt.Scene.from_file(scene_path("spheres.json"), random_spheres_seed=1)
    cam = sc.camera()
    sc.set_counters(True)
    sc.reset_stats()
    gpu_frame(sc, cam, 32, 24, 2, 8, seed=8)
    st = sc.stats()
    _, info = po.OracleScene(sc.desc()).render(cam, 32, 24, 2, 8, seed=8, rng="philox", counters=True)
    c = info["counters"]
    assert st.paths == 32 * 24 * 2
    n_march = int((sc.shape_kinds() == 3).sum())
    assert st.segments == c["segments"]
    assert st.segments * 8 < st.cull_tests < c["shape_tests"] // 2
    assert 0 < st.shape_tests < c["shape_tests"] // 4
    assert 0 < st.march_steps < c["march_steps"]
    assert st.kernel_launches > 0


def _load_named(name):
    """a fixture scene, or "march32": 32 ray-marched shapes, the most the wavefront marcher takes (bit 31 of its mask)"""
    if name == "march32":
        import json
        from test_gpu_frame_edges import marched_scene
        return rt.Scene.from_json(json.dumps(marched_scene(32)), add_random_spheres=False)
    return rt.Scene.from_file(scene_path(name), random_spheres_seed=1)


@pytest.mark.parametrize("name", ["spheres.json", "cornell_box.json", "dupin.json", "detached_materials.json",
                                  "light_source.json", "march32"])
def test_alternative_schedules_give_the_same_frame(monkeypatch, name):
    """the result does not depend on how the work is scheduled: the fused k_bounce (RT_B200_FUSED_BOUNCE), the
    linear scan without the cull tree (RT_B200_NO_CULL_TREE), the literal marching loop (RT_B200_NO_MARCH_SKIP), the
    flat list without its staged records (RT_B200_NO_FLAT_REC) and k_shade with and without its binned queue
    (RT_B200_SHADE_BINNED) reproduce the default wavefront frame (k_extend, k_march_filter, k_march, k_shade) bit for
    bit.
    The fused k_bounce draws random_in_unit_sphere with the sequential rejection loop and the default k_shade
    warp-cooperatively, so this also pins the cooperative sampler to the sequential one"""
    w, h, spp, depth, seed = 96, 72, 4, 8, 21
    sc = _load_named(name)
    ref = gpu_frame(sc, sc.camera(), w, h, spp, depth, seed)
    for var, val in (("RT_B200_FUSED_BOUNCE", "1"),
                     ("RT_B200_NO_CULL_TREE", "1"), ("RT_B200_NO_MARCH_SKIP", "1"), ("RT_B200_NO_FLAT_REC", "1"),
                     ("RT_B200_SHADE_BINNED", "1"), ("RT_B200_SHADE_BINNED", "0")):
        monkeypatch.setenv(var, val)
        alt = _load_named(name)
        got = gpu_frame(alt, alt.camera(), w, h, spp, depth, seed)
        monkeypatch.delenv(var)
        assert np.array_equal(got, ref), var


def test_binned_shade_queue_gives_the_same_frame_on_all_material_and_texture_branches(monkeypatch):
    """config 4b (every material / texture kind live): k_shade with its slots binned by (material kind, texture kind)
    -- the shade queue keyed by material -- against the arrival-order k_shade, bit for bit, at a size where a block's
    chunk of 1024 slots holds many keys"""
    frames = {}
    for binned in ("0", "1"):
        monkeypatch.setenv("RT_B200_SHADE_BINNED", binned)
        sc = rt.Scene.from_file(scene_path("detached_materials.json"), random_spheres_seed=1)
        cam = _variant_4b(sc)
        frames[binned] = gpu_frame(sc, cam, 320, 180, 8, 8, seed=17)
        monkeypatch.delenv("RT_B200_SHADE_BINNED")
    assert np.array_equal(frames["0"], frames["1"])
    assert frames["1"].mean() > 0.05


def test_distributed_renderer_frames_follow_their_parameters():
    """DistributedRenderer (world size 1 in-process; every GPU of the box under torchrun when there are several):
    a sequence of frames with CHANGING sample counts, rendered back to back, each equal to the unsharded frame.
    Identical consecutive frames cannot show a frame assembled / copied before its shards arrived; this can."""
    import subprocess
    import sys
    torch = pytest.importorskip("torch")
    tool = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools", "check_distributed_frames.py")
    n = min(torch.cuda.device_count(), 8)
    cmd = [sys.executable, tool] if n < 2 else [
        sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr", "127.0.0.1",
        "--master-port", "29547", tool]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert "deviating pixels 0" in r.stdout
