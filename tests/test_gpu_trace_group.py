"""rt_trace_pixel_samples_group[_device] (renderer::trace_pixel_samples_group, src/renderer/mod.rs:127-149): caller
rays of many pixels in one wavefront.

Group g = rays[offsets[g]:offsets[g+1]] are samples 0, 1, ... of pixel pixel_index[g]; its mean must be the oracle's
per-ray colours of those rays averaged as the device averages them, within one float ulp per path (check_groups in
tests/test_gpu_caller_rays.py: the same Philox paths, each rounded to float once), the one-pixel entry's result bit for bit, and -- fed the camera's own primary rays -- the rt_render_start frame bit for bit, whatever
the batch size, the lanes, the fused fallback or the order / split of the groups.
"""
import ctypes as C

import numpy as np
import pytest

import rs_pathtracing_b200 as rt
from rs_pathtracing_b200 import _ffi, api
from oracle import pyoracle as po

from conftest import scene_path

pytestmark = pytest.mark.gpu

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


def _group_rays(rng, cam, w, h, pixel, n):
    """n rays for pixel `pixel`: camera rays jittered inside the pixel, and unit directions drawn at random from the
    camera position"""
    x, y = pixel % w, pixel // w
    out = np.empty((n, 6))
    for k in range(n):
        if rng.random() < 0.6:
            u, v = rng.uniform(0, 1, 2)
            out[k] = po.get_ray(cam, w, h, x + u, y + v)
        else:
            d = rng.normal(size=3)
            out[k, :3] = cam.position.tuple()
            out[k, 3:] = d / np.linalg.norm(d)
    return out


def _groups(cam, sizes, seed, w=160, h=120):
    """rays, offsets, pixel_index for groups of the given sizes; the last two groups repeat a pixel index (with other
    rays), and a copy of group 2 (same rays, same pixel) is appended"""
    rng = np.random.default_rng(seed)
    sizes = list(sizes)
    pix = rng.integers(0, w * h, len(sizes)).astype(np.uint32)
    pix[-1] = pix[-2] = pix[0]
    rays = [_group_rays(rng, cam, w, h, int(p), n) for p, n in zip(pix, sizes)]
    rays.append(rays[2].copy())
    pix = np.append(pix, pix[2]).astype(np.uint32)
    sizes.append(sizes[2])
    offsets = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    return np.concatenate(rays).reshape(-1, 6), offsets, pix


def _split(rays, offsets, g):
    return rays[int(offsets[g]):int(offsets[g + 1])]


ORACLE_CASES = [("spheres.json", ""), ("cornell_box.json", ""), ("dupin.json", ""), ("detached_materials.json", "4b")]


@pytest.mark.parametrize("name,variant", ORACLE_CASES)
def test_group_means_match_oracle(name, variant):
    sc, cam = _load(name, variant)
    rng = np.random.default_rng(3)
    sizes = [1, 3, 10, 257, 0] + list(rng.integers(0, 40, 12)) + [0, 5, 5]
    rays, offsets, pix = _groups(cam, sizes, seed=11)
    depth, seed = 8, 77
    got = sc.trace_pixel_samples_group(rays, offsets, pix, depth, seed=seed)
    assert got.shape == (len(pix), 3)
    from test_gpu_caller_rays import check_groups   # (that module imports this one)
    cols = po.OracleScene(sc.desc()).group_sample_colors(rays, offsets, pix, depth, seed)
    check_groups(got, cols, offsets, f"{name}{variant} group means")
    assert np.array_equal(got[-1], got[2])    # identical rays, identical pixel index: identical means


@pytest.mark.parametrize("name,variant", [("spheres.json", ""), ("dupin.json", "")])
def test_every_group_equals_the_one_pixel_entry(name, variant):
    sc, cam = _load(name, variant)
    rays, offsets, pix = _groups(cam, [1, 3, 10, 257, 2, 31, 7, 7], seed=5)
    depth, seed = 8, 3
    got = sc.trace_pixel_samples_group(rays, offsets, pix, depth, seed=seed)
    for g in range(len(pix)):
        one = sc.trace_pixel_samples(_split(rays, offsets, g), depth, seed=seed, pixel_index=int(pix[g]))
        assert np.array_equal(got[g], one), g


def _primary_rays(cam, w, h, spp, seed):
    """the frame's own primary rays: MultisamplerRayCaster::next with the Philox draws of event 0"""
    rays = np.empty((w * h * spp, 6))
    k = 0
    for y in range(h):
        for x in range(w):
            for s in range(spp):
                u, v = po.philox_stream(seed, x + y * w, s, 0, 2)
                rays[k] = po.get_ray(cam, w, h, x + u, y + v)
                k += 1
    return rays


@pytest.mark.parametrize("name,w,h", [("spheres.json", 64, 48), ("cornell_box.json", 48, 48)])
def test_camera_rays_reproduce_the_frame(name, w, h):
    spp, depth, seed = 4, 8, 1234
    sc, cam = _load(name)
    rays = _primary_rays(cam, w, h, spp, seed)
    offsets = np.arange(0, w * h * spp + 1, spp, dtype=np.uint64)
    pix = np.arange(w * h, dtype=np.uint32)
    got = sc.trace_pixel_samples_group(rays, offsets, pix, depth, seed=seed)
    frame = rt.GpuRenderer(sc, 12, depth, seed=seed).render(cam, w, h, spp)
    assert np.array_equal(got, frame.reshape(-1, 3))


def test_results_do_not_depend_on_the_schedule(monkeypatch):
    """batch sizes that split groups over batches (one group of 5000 rays, one of exactly a batch), 1 to 3 lanes, the
    fused k_bounce fallback, another group order and two calls instead of one: the same means, bit for bit"""
    name = "spheres.json"
    sc, cam = _load(name)
    rng = np.random.default_rng(8)
    sizes = list(rng.integers(0, 30, 40)) + [5000, 0, 0, 1000, 999, 1001] + list(rng.integers(0, 300, 20))
    rays, offsets, pix = _groups(cam, sizes, seed=2)
    depth, seed = 8, 41
    ref = sc.trace_pixel_samples_group(rays, offsets, pix, depth, seed=seed)
    assert np.isfinite(ref[np.diff(offsets) > 0]).all()

    def run(env):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        alt, _ = _load(name)   # a new device handle reads the variables
        got = alt.trace_pixel_samples_group(rays, offsets, pix, depth, seed=seed)
        for k in env:
            monkeypatch.delenv(k)
        return got

    for env in ({"RT_B200_BATCH_PATHS": "1000"}, {"RT_B200_BATCH_PATHS": "4096"},
                {"RT_B200_BATCH_PATHS": "1000", "RT_B200_LANES": "1"},
                {"RT_B200_BATCH_PATHS": "1000", "RT_B200_LANES": "2"},
                {"RT_B200_BATCH_PATHS": "1000", "RT_B200_LANES": "3"},
                {"RT_B200_FUSED_BOUNCE": "1"}, {"RT_B200_FUSED_BOUNCE": "1", "RT_B200_BATCH_PATHS": "1000"}):
        assert np.array_equal(run(env), ref, equal_nan=True), env

    # another order of the groups, in two calls
    perm = np.random.default_rng(1).permutation(len(pix))
    parts = [perm[: len(perm) // 2], perm[len(perm) // 2:]]
    got = np.empty_like(ref)
    for part in parts:
        r = np.concatenate([_split(rays, offsets, g) for g in part]).reshape(-1, 6)
        off = np.concatenate([[0], np.cumsum(np.diff(offsets)[part])]).astype(np.uint64)
        got[part] = sc.trace_pixel_samples_group(r, off, pix[part], depth, seed=seed)
    assert np.array_equal(got, ref, equal_nan=True)


def test_device_form_on_torch_streams():
    """rays in a torch tensor written on a non-default stream, the call inside torch.cuda.stream(s): the result equals
    the host form bit for bit; the same on torch's default (legacy) stream"""
    torch = pytest.importorskip("torch")
    sc, cam = _load("cornell_box.json")
    rng = np.random.default_rng(4)
    rays, offsets, pix = _groups(cam, list(rng.integers(0, 50, 200)) + [0, 3000], seed=6)
    depth, seed = 8, 9
    want = sc.trace_pixel_samples_group(rays, offsets, pix, depth, seed=seed)
    src = torch.from_numpy(rays).pin_memory()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        t = torch.empty((rays.shape[0], 6), dtype=torch.float64, device="cuda")
        t.copy_(src, non_blocking=True)
        t.mul_(1.0)
        means = sc.trace_pixel_samples_group(t, offsets, pix, depth, seed=seed)
        del t                          # the caching allocator may hand the rays' memory to the next op on s
        junk = torch.full((rays.shape[0], 6), 7.0, dtype=torch.float64, device="cuda")
        got = means.cpu().numpy()
    s.synchronize()
    assert isinstance(means, torch.Tensor) and means.device.type == "cuda" and means.dtype == torch.float64
    assert np.array_equal(got, want, equal_nan=True)
    del junk
    t2 = torch.from_numpy(rays).cuda()
    got2 = sc.trace_pixel_samples_group(t2, offsets, pix, depth, seed=seed)
    assert np.array_equal(got2.cpu().numpy(), want, equal_nan=True)
    assert sc.trace_pixel_samples_group(t2[:0], [0], [], depth, seed=seed).shape == (0, 3)


def test_state_is_left_alone():
    w, h, depth, seed = 64, 48, 8, 9
    sc, cam = _load("cornell_box.json")
    other, _ = _load("cornell_box.json")
    ref8 = rt.GpuRenderer(other, 12, depth, seed=seed).render(cam, w, h, 8)
    rays, offsets, pix = _groups(cam, [1, 3, 10, 257, 0, 20], seed=1)
    ds = sc.device_scene(0)
    # progressive accumulation: 4 spp, a group call, 4 spp more = the 8-spp frame
    api.render_set_accumulate(ds, True)
    buf = np.zeros((h, w, 3))
    api.render_start(ds, cam, api.render_params(w, h, 4, depth, seed))
    api.render_wait(ds, buf)
    sc.reset_stats()
    sc.trace_pixel_samples_group(rays, offsets, pix, depth, seed=seed)
    assert sc.stats().paths == rays.shape[0]
    api.render_start(ds, cam, api.render_params(w, h, 4, depth, seed))
    api.render_wait(ds, buf)
    assert api.render_accumulated_samples(ds) == 8
    assert np.array_equal(buf, ref8)
    api.render_set_accumulate(ds, False)
    # a frame in flight
    api.render_start(ds, cam, api.render_params(w, h, 2, depth, seed))
    with pytest.raises(rt.RtError, match="in flight"):
        sc.trace_pixel_samples_group(rays, offsets, pix, depth, seed=seed)
    api.render_wait(ds, buf)


def _raw_group(handle, rays, n_rays, offsets, pix, n_groups, depth, seed, means):
    p = lambda a: a.ctypes.data_as(C.c_void_p) if a is not None else None
    return _ffi.core().rt_trace_pixel_samples_group(handle, p(rays), n_rays, p(offsets), p(pix), n_groups, depth, seed,
                                                    p(means))


def test_multi_device_handle_addresses_its_first_device():
    n_dev = rt.device_count()
    if n_dev < 2:
        pytest.skip("needs two GPUs")
    sc, cam = _load("spheres.json")
    rays, offsets, pix = _groups(cam, [1, 3, 10, 257, 0, 20], seed=1)
    want = sc.trace_pixel_samples_group(rays, offsets, pix, 8, seed=2)
    multi, _ = _load("spheres.json")
    h = multi.device_scene_multi(list(range(n_dev)))
    got = np.empty_like(want)
    api._check(_raw_group(h, rays, rays.shape[0], offsets, pix, len(pix), 8, 2, got))
    assert np.array_equal(got, want, equal_nan=True)


def test_bad_input_is_rejected():
    sc, cam = _load("cube_test.json")
    rays, offsets, pix = _groups(cam, [2, 3, 4], seed=1)
    depth = 8
    assert list(offsets) == [0, 2, 5, 9, 13]
    bad_offsets = ([1, 2, 5, 9, 13], [0, 3, 2, 9, 13], [0, 2, 5, 9, 12])   # offsets[0] != 0, decreasing, end != n_rays
    for off in bad_offsets:
        with pytest.raises(rt.RtError, match="-1"):
            sc.trace_pixel_samples_group(rays, off, pix, depth)
    with pytest.raises(rt.RtError, match="-1"):
        sc.trace_pixel_samples_group(rays, offsets, pix, 63)
    assert sc.trace_pixel_samples_group(rays, offsets, pix, 62).shape == (len(pix), 3)
    h = sc.device_scene()
    means = np.empty((len(pix), 3))
    n = rays.shape[0]
    off = np.asarray(offsets, np.uint64)
    # a group of 2^32 rays (rejected from the offsets alone, before any ray is read)
    big = np.array([0, 1 << 32], np.uint64)
    assert _raw_group(h, rays, 1 << 32, big, pix[:1], 1, depth, 0, means) == _ffi.RT_ERR_INVALID
    # NULL arrays where something is needed
    assert _raw_group(h, None, n, off, pix, len(pix), depth, 0, means) == _ffi.RT_ERR_INVALID
    assert _raw_group(h, rays, n, None, pix, len(pix), depth, 0, means) == _ffi.RT_ERR_INVALID
    assert _raw_group(h, rays, n, off, None, len(pix), depth, 0, means) == _ffi.RT_ERR_INVALID
    assert _raw_group(h, rays, n, off, pix, len(pix), depth, 0, None) == _ffi.RT_ERR_INVALID
    assert _ffi.core().rt_trace_pixel_samples_group_device(h, None, n, off.ctypes.data_as(C.c_void_p),
                                                           pix.ctypes.data_as(C.c_void_p), len(pix), depth, 0, None,
                                                           None) == _ffi.RT_ERR_INVALID
    # no groups: nothing to do
    assert sc.trace_pixel_samples_group(np.zeros((0, 6)), [0], [], depth).shape == (0, 3)
    assert _raw_group(h, None, 0, None, None, 0, depth, 0, None) == _ffi.RT_OK
