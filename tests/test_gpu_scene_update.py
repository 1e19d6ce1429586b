"""Scene updates on live handles, bit for bit against fresh handles of the edited description.

rt_scene_update replaces the whole scene (any table sizes, the wavefront / fused switch, the shade-bin policy);
rt_scene_update_transforms moves shapes and refits the cull tree in place.  Either way every entry point of the updated
handle must give what a handle created from the edited description gives: the nearest hits (BRUTE and FAST, every
output, and RT_ISECT_VERIFY's self-check), frames, views, counts and adaptive frames and caller-ray groups."""
import ctypes as C
import json
import zlib

import numpy as np
import pytest

import rs_pathtracing_b200 as rt
from rs_pathtracing_b200 import _ffi, api
from oracle import pyoracle as po

from conftest import scene_path
from test_gpu_frame_edges import check_frame, marched_scene
from test_gpu_render import _variant_4b

pytestmark = pytest.mark.gpu

W, H, SPP, DEPTH, SEED = 48, 36, 3, 6, 11


def p(a):
    return a.ctypes.data_as(C.c_void_p)


class Edited:
    """a host scene's description with its own, editable copies of the inverse and direct rows"""

    def __init__(self, sc):
        self.sc = sc
        d = sc.desc()
        self.inv = np.ctypeslib.as_array(d.inverse, shape=(d.n_shapes, 12)).copy() if d.n_shapes else np.zeros((0, 12))
        self.dir = np.ctypeslib.as_array(d.direct, shape=(d.n_shapes, 12)).copy() if d.n_shapes else np.zeros((0, 12))

    def desc(self):
        d = self.sc.desc()
        if d.n_shapes:
            d.inverse = self.inv.ctypes.data_as(C.POINTER(C.c_double))
            d.direct = self.dir.ctypes.data_as(C.POINTER(C.c_double))
        return d

    def move(self, rng, index, step):
        for i in index:
            shift = rng.normal(0.0, step, 3)
            m = self.inv[i].reshape(3, 4)
            m[:, 3] -= m[:, :3] @ shift
            self.dir[i].reshape(3, 4)[:, 3] += shift
        return self.inv[index].copy(), self.dir[index].copy()


def create(desc):
    h = C.c_void_p()
    rc = _ffi.core().rt_scene_create(C.byref(desc), 0, C.byref(h))
    assert rc == 0, _ffi.core().rt_last_error()
    return h


def update_transforms(h, index, inv, direct):
    api.update_transforms(h, np.asarray(index, np.uint32), inv, direct)


def probe_rays(cam, n=4096, seed=0):
    rng = np.random.default_rng(seed)
    xy = rng.uniform(0, 1, (n, 2)) * (W, H)
    return np.array([po.get_ray(cam, W, H, x, y) for x, y in xy])


def intersect(h, rays, mode):
    n = len(rays)
    out = dict(index=np.empty(n, np.int32), t=np.empty(n), normal=np.empty((n, 3)), point=np.empty((n, 3)),
               uv=np.empty((n, 2)), ff=np.empty(n, np.uint8))
    rays = np.ascontiguousarray(rays, np.float64)
    rc = _ffi.core().rt_intersect_batch(h, p(rays), n, 0.001, np.inf, mode, p(out["index"]), p(out["t"]),
                                        p(out["normal"]), p(out["point"]), p(out["uv"]), p(out["ff"]))
    assert rc == 0, _ffi.core().rt_last_error()
    return out


def frame(h, cam, spp=SPP, seed=SEED):
    api.render_start(h, cam, api.render_params(W, H, spp, DEPTH, seed))
    buf = np.empty((H, W, 3))
    api.render_wait(h, buf)
    return buf


def results(h, cam, wavefront=True):
    """everything the handle computes for one camera, as a dict of arrays"""
    rays = probe_rays(cam)
    out = {}
    for mode in (rt.RT_ISECT_BRUTE, rt.RT_ISECT_FAST):
        for k, v in intersect(h, rays, mode).items():
            out[f"isect{mode}_{k}"] = v
    out["frame"] = frame(h, cam)
    cam2 = rt.camera_new(np.array(cam.position.tuple()) * 1.1, (-cam.position.x, -cam.position.y, -cam.position.z),
                         (0, 1, 0), 1.0, cam.fov_rad)
    api.render_start_views(h, [cam, cam2], api.render_params(W, H, 2, DEPTH, SEED))
    views = np.empty((2, H, W, 3))
    api.render_wait(h, views)
    out["views"] = views
    counts = (np.arange(W * H, dtype=np.uint32) % 4).reshape(H, W)
    api.render_start_counts(h, cam, api.render_params(W, H, 3, DEPTH, SEED), counts)
    cf = np.empty((H, W, 3))
    api.render_wait(h, cf)
    out["counts"] = cf
    if wavefront:
        api.render_start_adaptive(h, cam, api.render_params(W, H, 8, DEPTH, SEED), 2, 0.05)
        af = np.empty((H, W, 3))
        api.render_wait(h, af)
        out["adaptive"] = af
    gr = probe_rays(cam, 600, seed=1)
    offsets = np.array([0, 1, 1, 100, 350, 600], np.uint64)
    pix = np.array([5, 9, 9, 1000, 3], np.uint32)
    means = np.empty((5, 3))
    rc = _ffi.core().rt_trace_pixel_samples_group(h, p(np.ascontiguousarray(gr)), 600, p(offsets), p(pix), 5, DEPTH, SEED,
                                                  p(means))
    assert rc == 0, _ffi.core().rt_last_error()
    out["groups"] = means
    return out


def assert_same(a, b, what):
    assert a.keys() == b.keys()
    for k in a:
        assert np.array_equal(a[k], b[k], equal_nan=True), f"{what}: {k} differs"


def verify_clean(h, rays):
    core = _ffi.core()
    core.rt_reset_stats(h)
    intersect(h, rays, rt.RT_ISECT_VERIFY)
    st = rt.Stats()
    assert core.rt_get_stats(h, C.byref(st)) == 0
    return st.verify_rays, st.verify_false_culls


def load(name):
    if name in ("march32", "march33"):
        sc = rt.Scene.from_json(json.dumps(marched_scene(int(name[5:]))), add_random_spheres=False)
        return sc, sc.camera()
    if name == "4b":
        sc = rt.Scene.from_file(scene_path("detached_materials.json"), random_spheres_seed=1)
        return sc, _variant_4b(sc)
    sc = rt.Scene.from_file(scene_path(name), random_spheres_seed=1)
    cam = sc.camera() if name != "empty.json" else rt.Scene.from_file(scene_path("spheres.json")).camera()
    return sc, cam


def test_full_updates_cycle_through_scenes():
    """one handle goes spheres -> cornell_box -> dupin -> cfg 4b -> march33 (the fused fallback) -> march32 (back to the
    wavefront) -> empty -> spheres; after every step it equals a fresh handle of that scene"""
    sc0, _ = load("spheres.json")
    h = create(sc0.desc())
    try:
        for name in ("cornell_box.json", "dupin.json", "4b", "march33", "march32", "empty.json", "spheres.json"):
            sc, cam = load(name)
            api.scene_update(h, sc.desc())
            fresh = create(sc.desc())
            try:
                wavefront = name != "march33"
                assert_same(results(h, cam, wavefront), results(fresh, cam, wavefront), name)
            finally:
                _ffi.core().rt_scene_destroy(fresh)
    finally:
        _ffi.core().rt_scene_destroy(h)


@pytest.mark.parametrize("name,what", [("spheres.json", 1), ("spheres.json", 16), ("spheres.json", 481),
                                       ("cornell_box.json", "all"), ("dupin.json", "all"), ("torus.json", "all"),
                                       ("march32", "all")])
def test_transform_updates_equal_a_fresh_handle(name, what):
    """random motions of 1, 16 and 481 spheres, of every shape of cornell_box (Rectangles, Cubes), dupin and march32
    (ray-marched shapes) and torus.json"""
    sc, cam = load(name)
    ed = Edited(sc)
    n = len(ed.inv)
    rng = np.random.default_rng(zlib.crc32(f"{name} {what}".encode()))
    h = create(ed.desc())
    try:
        for step in (0.05, 0.5):
            if what == "all":
                index = np.arange(n)
            else:
                spheres = np.flatnonzero(sc.shape_kinds() == _ffi.RT_SHAPE_SPHERE)
                index = rng.choice(spheres, size=min(what, len(spheres)), replace=False)
            update_transforms(h, index, *ed.move(rng, index, step))
            fresh = create(ed.desc())
            try:
                assert_same(results(h, cam), results(fresh, cam), f"{name} {what} step {step}")
            finally:
                _ffi.core().rt_scene_destroy(fresh)
    finally:
        _ffi.core().rt_scene_destroy(h)


def test_verify_after_100_refits():
    """100 successive random-walk refits of 16 spheres each: RT_ISECT_VERIFY finds no disagreement and no false cull on
    1 Mi rays, and the nearest hits equal a fresh handle's"""
    sc, cam = load("spheres.json")
    ed = Edited(sc)
    rng = np.random.default_rng(3)
    spheres = np.flatnonzero(sc.shape_kinds() == _ffi.RT_SHAPE_SPHERE)
    h = create(ed.desc())
    try:
        for _ in range(100):
            index = rng.choice(spheres, size=16, replace=False)
            update_transforms(h, index, *ed.move(rng, index, 0.2))
        o = rng.uniform(-15, 15, (1 << 20, 3)) + (0, 8, 0)
        rays = rt.make_rays(o, rng.uniform(-6, 6, (1 << 20, 3)) - o)
        assert verify_clean(h, rays) == (0, 0)
        fresh = create(ed.desc())
        try:
            for mode in (rt.RT_ISECT_BRUTE, rt.RT_ISECT_FAST):
                a, b = intersect(h, rays[:1 << 18], mode), intersect(fresh, rays[:1 << 18], mode)
                for k in a:
                    assert np.array_equal(a[k], b[k], equal_nan=True), k
        finally:
            _ffi.core().rt_scene_destroy(fresh)
    finally:
        _ffi.core().rt_scene_destroy(h)


@pytest.mark.parametrize("case", ["far", "shrunk", "ill_conditioned", "singular"])
def test_extreme_motions_and_back(case):
    sc, cam = load("spheres.json")
    ed = Edited(sc)
    rng = np.random.default_rng(4)
    index = rng.choice(np.flatnonzero(sc.shape_kinds() == _ffi.RT_SHAPE_SPHERE)[5:], size=16, replace=False)
    back_inv, back_dir = ed.inv[index].copy(), ed.dir[index].copy()
    for k, i in enumerate(index):
        c = ed.dir[i].reshape(3, 4)[:, 3]
        t = {"far": (c + rng.normal(0, 1e6, 3), (0, 0, 0), (0.2, 0.2, 0.2)),
             "shrunk": (c, (0, 0, 0), (2e-7,) * 3),
             "ill_conditioned": (c, (10, 20, 30), (0.2, 0.2, 20.0)),
             "singular": (c, (0, 0, 0), (0.2, 0.0, 0.2))}[case]
        ed.inv[i], ed.dir[i] = api.transform(*t)
    h = create(sc.desc())
    try:
        for inv, direct in ((ed.inv[index].copy(), ed.dir[index].copy()), (back_inv, back_dir)):
            update_transforms(h, index, inv, direct)
            ed.inv[index], ed.dir[index] = inv, direct
            fresh = create(ed.desc())
            try:
                assert_same(results(h, cam), results(fresh, cam), case)
            finally:
                _ffi.core().rt_scene_destroy(fresh)
            rays = probe_rays(cam, 1 << 16, seed=5)
            assert verify_clean(h, rays) == (0, 0)
    finally:
        _ffi.core().rt_scene_destroy(h)


def test_frame_after_edits_matches_the_oracle():
    sc, cam = load("cornell_box.json")
    ed = Edited(sc)
    rng = np.random.default_rng(9)
    h = create(ed.desc())
    try:
        index = rng.choice(len(ed.inv), size=40, replace=False)
        update_transforms(h, index, *ed.move(rng, index, 0.3))
        got = frame(h, cam, spp=2)
        check_frame(got, po.OracleScene(ed.desc()), cam, W, H, 2, DEPTH, SEED, "cornell_box after edits")
    finally:
        _ffi.core().rt_scene_destroy(h)


def test_state_rules():
    core = _ffi.core()
    sc, cam = load("spheres.json")
    ed = Edited(sc)
    old = Edited(sc)
    rng = np.random.default_rng(10)
    h = create(ed.desc())
    try:
        # in flight: RT_ERR_STATE, and the frame in flight is the old scene's
        ref_old = frame(h, cam)
        api.render_start(h, cam, api.render_params(W, H, SPP, DEPTH, SEED))
        index = np.arange(20, 60)
        inv, direct = ed.move(rng, index, 0.5)
        assert core.rt_scene_update_transforms(h, len(index), p(index.astype(np.uint32)), p(inv), p(direct)) == _ffi.RT_ERR_STATE
        assert core.rt_scene_update(h, C.byref(ed.desc())) == _ffi.RT_ERR_STATE
        buf = np.empty((H, W, 3))
        api.render_wait(h, buf)
        assert np.array_equal(buf, ref_old)
        # the last frame stays readable after an update
        rgba_before = api.tonemap_last_frame(h)
        update_transforms(h, index, inv, direct)
        assert np.array_equal(api.tonemap_last_frame(h), rgba_before)
        # a failed update leaves the (new) scene rendering bit for bit
        ref_new = frame(h, cam)
        bad = ed.desc()
        mats = np.ctypeslib.as_array(bad.material, shape=(bad.n_shapes,)).copy()
        mats[0] = bad.n_materials
        bad.material = mats.ctypes.data_as(C.POINTER(C.c_uint32))
        assert core.rt_scene_update(h, C.byref(bad)) == _ffi.RT_ERR_INVALID
        assert np.array_equal(frame(h, cam), ref_new)
        fresh = create(ed.desc())
        assert np.array_equal(frame(fresh, cam), ref_new)
        core.rt_scene_destroy(fresh)
        # accumulation restarts after an update
        assert core.rt_render_set_accumulate(h, 1) == 0
        frame(h, cam)
        frame(h, cam)
        n = C.c_uint32()
        core.rt_render_accumulated_samples(h, C.byref(n))
        assert n.value == 2 * SPP
        back = np.arange(20, 60)
        update_transforms(h, back, old.inv[back], old.dir[back])
        core.rt_render_accumulated_samples(h, C.byref(n))
        assert n.value == 0
        assert np.array_equal(frame(h, cam), ref_old)
        core.rt_render_set_accumulate(h, 0)
    finally:
        core.rt_scene_destroy(h)


def test_updates_are_ordered_against_caller_streams():
    """rt_intersect_batch_device / rt_trace_pixel_samples_group_device queued on a torch stream before an update see the
    old scene, calls after it the new one"""
    torch = pytest.importorskip("torch")
    sc, cam = load("spheres.json")
    ed = Edited(sc)
    rng = np.random.default_rng(11)
    rays = probe_rays(cam, 1 << 16, seed=6)
    h = create(ed.desc())
    try:
        core = _ffi.core()
        n_g = 4096   # groups of 16 rays
        offsets = np.arange(0, len(rays) + 1, 16, dtype=np.uint64)[:n_g + 1]
        pix = np.arange(n_g, dtype=np.uint32)
        g_rays = np.ascontiguousarray(rays[:16 * n_g])

        def groups_host(hd):
            means = np.empty((n_g, 3))
            assert core.rt_trace_pixel_samples_group(hd, p(g_rays), len(g_rays), p(offsets), p(pix), n_g, DEPTH, SEED,
                                                     p(means)) == 0
            return means

        old_hits = intersect(h, rays, rt.RT_ISECT_FAST)["index"]
        old_means = groups_host(h)
        index = np.flatnonzero(sc.shape_kinds() == _ffi.RT_SHAPE_SPHERE)[:200]
        inv, direct = ed.move(rng, index, 2.0)
        fresh = create(ed.desc())
        new_hits = intersect(fresh, rays, rt.RT_ISECT_FAST)["index"]
        new_means = groups_host(fresh)
        core.rt_scene_destroy(fresh)
        assert not np.array_equal(old_hits, new_hits) and not np.array_equal(old_means, new_means)
        s = torch.cuda.Stream()
        d_rays = torch.from_numpy(np.ascontiguousarray(rays)).cuda()
        d_grays = torch.from_numpy(g_rays).cuda()
        before = torch.empty(len(rays), dtype=torch.int32, device="cuda")
        after = torch.empty_like(before)
        m_before = torch.empty((n_g, 3), dtype=torch.float64, device="cuda")
        m_after = torch.empty_like(m_before)
        cs = C.c_void_p(s.cuda_stream)
        with torch.cuda.stream(s):
            for _ in range(8):   # enough work queued that the update would overtake it if it were not ordered
                assert core.rt_intersect_batch_device(h, d_rays.data_ptr(), len(rays), 0.001, np.inf, rt.RT_ISECT_BRUTE,
                                                      before.data_ptr(), None, None, None, None, None, cs) == 0
            assert core.rt_trace_pixel_samples_group_device(h, d_grays.data_ptr(), len(g_rays), p(offsets), p(pix), n_g,
                                                            DEPTH, SEED, m_before.data_ptr(), cs) == 0
            update_transforms(h, index, inv, direct)
            assert core.rt_intersect_batch_device(h, d_rays.data_ptr(), len(rays), 0.001, np.inf, rt.RT_ISECT_FAST,
                                                  after.data_ptr(), None, None, None, None, None, cs) == 0
            assert core.rt_trace_pixel_samples_group_device(h, d_grays.data_ptr(), len(g_rays), p(offsets), p(pix), n_g,
                                                            DEPTH, SEED, m_after.data_ptr(), cs) == 0
        s.synchronize()
        assert np.array_equal(before.cpu().numpy(), old_hits)
        assert np.array_equal(after.cpu().numpy(), new_hits)
        assert np.array_equal(m_before.cpu().numpy(), old_means)
        assert np.array_equal(m_after.cpu().numpy(), new_means)
    finally:
        _ffi.core().rt_scene_destroy(h)


def test_multi_device_handle_updates_every_device():
    if rt.device_count() < 2:
        pytest.skip("needs two devices")
    sc, cam = load("spheres.json")
    ed = Edited(sc)
    rng = np.random.default_rng(12)
    ids = (C.c_int * 2)(0, 1)
    h = C.c_void_p()
    assert _ffi.core().rt_scene_create_multi(C.byref(ed.desc()), 2, ids, C.byref(h)) == 0
    try:
        index = rng.choice(len(ed.inv), size=100, replace=False)
        update_transforms(h, index, *ed.move(rng, index, 0.5))
        fresh = create(ed.desc())
        try:
            assert np.array_equal(frame(h, cam), frame(fresh, cam))
        finally:
            _ffi.core().rt_scene_destroy(fresh)
    finally:
        _ffi.core().rt_scene_destroy(h)


def test_transforms_on_a_scene_with_levels_above_the_roots():
    """10^4 shapes (one level of nodes above the roots, so the refit writes upper nodes too): every shape of a third of
    the tree moved, nearest hits BRUTE and FAST with every output equal to a fresh handle's, RT_ISECT_VERIFY clean"""
    from test_cull_cpu import big_scene, box_rays
    sc = big_scene(10000, seed=5, extent=25.0)
    d = sc.desc()
    counts = [C.c_uint32() for _ in range(4)]
    worst = C.c_double()
    assert _ffi.core().rt_cull_tree_check(C.byref(d), *[C.byref(x) for x in counts], C.byref(worst)) == 0
    assert counts[0].value > 8   # more than 8 roots: at least one level above them
    ed = Edited(sc)
    rng = np.random.default_rng(13)
    h = create(ed.desc())
    try:
        rays = box_rays(1 << 16, seed=14, extent=25.0)
        for step in (0.2, 3.0):
            index = rng.choice(len(ed.inv), size=3500, replace=False)
            update_transforms(h, index, *ed.move(rng, index, step))
        fresh = create(ed.desc())
        try:
            for mode in (rt.RT_ISECT_BRUTE, rt.RT_ISECT_FAST):
                a, b = intersect(h, rays, mode), intersect(fresh, rays, mode)
                for k in a:
                    assert np.array_equal(a[k], b[k], equal_nan=True), (mode, k)
        finally:
            _ffi.core().rt_scene_destroy(fresh)
        assert verify_clean(h, rays) == (0, 0)
    finally:
        _ffi.core().rt_scene_destroy(h)


@pytest.mark.parametrize("lanes", ["1", "3"])
def test_transform_updates_frames_on_1_and_3_lanes(monkeypatch, lanes):
    """frames of many small batches over 1 and 3 lanes after transform updates == a fresh handle's"""
    monkeypatch.setenv("RT_B200_LANES", lanes)
    monkeypatch.setenv("RT_B200_BATCH_PATHS", "700")
    sc, cam = load("cornell_box.json")
    ed = Edited(sc)
    rng = np.random.default_rng(15)
    h = create(ed.desc())
    try:
        for _ in range(3):
            index = rng.choice(len(ed.inv), size=60, replace=False)
            update_transforms(h, index, *ed.move(rng, index, 0.3))
            fresh = create(ed.desc())
            try:
                assert np.array_equal(frame(h, cam), frame(fresh, cam))
            finally:
                _ffi.core().rt_scene_destroy(fresh)
    finally:
        _ffi.core().rt_scene_destroy(h)


def test_gpu_renderer_follows_scene_set_transforms():
    """GpuRenderer renders what its Scene holds when a frame starts: Scene.set_transforms between two frames moves the
    shapes in the renderer's handle, and the frame equals a fresh renderer's on a scene loaded with those transforms"""
    sc = rt.Scene.from_file(scene_path("spheres.json"), random_spheres_seed=1)
    cam = sc.camera()
    r = rt.GpuRenderer(sc, 12, DEPTH, seed=3)
    first = r.render(cam, W, H, SPP)
    n = sc.shape_count
    rng = np.random.default_rng(16)
    index = rng.choice(np.arange(5, n), size=40, replace=False)
    moves = [(rng.uniform(-4, 4, 3) * (1, 0, 1) + (0, 0.2, 0), (0, 0, 0), (0.2, 0.2, 0.2)) for _ in index]
    sc.set_transforms(index, [m[0] for m in moves], [m[1] for m in moves], [m[2] for m in moves])
    moved = r.render(cam, W, H, SPP)
    ref_sc = rt.Scene.from_file(scene_path("spheres.json"), random_spheres_seed=1)
    ref_sc.set_transforms(index, [m[0] for m in moves], [m[1] for m in moves], [m[2] for m in moves])
    ref = rt.GpuRenderer(ref_sc, 12, DEPTH, seed=3).render(cam, W, H, SPP)
    assert np.array_equal(moved, ref)
    assert not np.array_equal(moved, first)
    # the scene's description moved too: an oracle built from it agrees with the frame
    check_frame(moved, po.OracleScene(sc.desc()), cam, W, H, SPP, DEPTH, 3, "GpuRenderer after Scene.set_transforms")


def test_distributed_moving_object_sequence():
    """DistributedRenderer.render_jobs_device with per-job transforms (two frames in flight on two handles) and
    update_transforms == fresh handles frame by frame (tools/check_distributed_scene_update.py; every GPU of the box
    under torchrun)"""
    import os
    import subprocess
    import sys
    torch = pytest.importorskip("torch")
    tool = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools",
                        "check_distributed_scene_update.py")
    n = min(torch.cuda.device_count(), 8)
    cmd = [sys.executable, tool] if n < 2 else [
        sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr", "127.0.0.1",
        "--master-port", "29566", tool]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-2000:]
    assert "deviating frames 0" in res.stdout
