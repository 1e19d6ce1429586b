"""Scene updates on live handles without a device: argument checks of rt_scene_update / rt_scene_update_transforms and
the Python face, and the conservativeness of the cull-tree refit through rt_cull_refit_check (the host refit the
transforms entry runs, checked with rt_cull_tree_check's metric against every shape's true ball after the move)."""
import ctypes as C
import json
import zlib

import numpy as np
import pytest

import rs_pathtracing_b200 as rt
from rs_pathtracing_b200 import _ffi, api

from conftest import scene_path
from test_cull_cpu import big_scene
from test_gpu_intersect import TRIO

FIXTURES = ["spheres.json", "cornell_box.json", "detached_materials.json", "dupin.json", "cube_test.json",
            "light_source.json", "torus.json"]


def p(a):
    return a.ctypes.data_as(C.c_void_p)


def refit_worst(sc, index, inverse):
    d = sc.desc()
    index = np.ascontiguousarray(index, dtype=np.uint32)
    inverse = np.ascontiguousarray(inverse, dtype=np.float64)
    worst = C.c_double()
    rc = _ffi.core().rt_cull_refit_check(C.byref(d), len(index), p(index), p(inverse), C.byref(worst))
    assert rc == 0, _ffi.core().rt_last_error()
    return worst.value


def current_inverse(sc):
    d = sc.desc()
    return np.ctypeslib.as_array(d.inverse, shape=(d.n_shapes, 12)).copy()


def random_moves(rng, base, index, step):
    """each listed shape translated by a random step of size ~step (world space), scale and rotation kept"""
    inv = base[index].copy()
    for k in range(len(index)):
        m = inv[k].reshape(3, 4)
        shift = rng.normal(0.0, step, 3)
        m[:, 3] -= m[:, :3] @ shift   # inverse of (translate by shift) o T
    return inv


def test_entries_reject_null_arguments():
    core = _ffi.core()
    sc = rt.Scene.from_file(scene_path("spheres.json"), random_spheres_seed=1)
    d = sc.desc()
    idx = np.zeros(1, np.uint32)
    rows = np.zeros((1, 12))
    assert core.rt_scene_update(None, C.byref(d)) == _ffi.RT_ERR_INVALID
    assert core.rt_scene_update(None, None) == _ffi.RT_ERR_INVALID
    assert core.rt_scene_update_transforms(None, 1, p(idx), p(rows), p(rows)) == _ffi.RT_ERR_INVALID
    worst = C.c_double()
    assert core.rt_cull_refit_check(None, 0, None, None, C.byref(worst)) == _ffi.RT_ERR_INVALID
    assert core.rt_cull_refit_check(C.byref(d), 0, None, None, None) == _ffi.RT_ERR_INVALID
    assert core.rt_cull_refit_check(C.byref(d), 1, None, p(rows), C.byref(worst)) == _ffi.RT_ERR_INVALID
    assert core.rt_cull_refit_check(C.byref(d), 1, p(idx), None, C.byref(worst)) == _ffi.RT_ERR_INVALID
    assert core.rt_cull_refit_check(C.byref(d), 0, None, None, C.byref(worst)) == 0


def test_indices_out_of_range_or_twice_are_rejected():
    core = _ffi.core()
    sc = rt.Scene.from_file(scene_path("cornell_box.json"), random_spheres_seed=1)
    d = sc.desc()
    worst = C.c_double()
    for bad in ([d.n_shapes], [0, d.n_shapes + 7], [3, 5, 3], [2**32 - 1]):
        idx = np.array(bad, np.uint32)
        rows = np.tile(current_inverse(sc)[0], (len(bad), 1))
        assert core.rt_cull_refit_check(C.byref(d), len(idx), p(idx), p(rows), C.byref(worst)) == _ffi.RT_ERR_INVALID
    idx = np.array([d.n_shapes - 1, 0], np.uint32)
    assert core.rt_cull_refit_check(C.byref(d), 2, p(idx), p(current_inverse(sc)[[d.n_shapes - 1, 0]]),
                                    C.byref(worst)) == 0


def test_invalid_description_is_rejected_before_any_device_work():
    """rt_scene_update checks the description first, like rt_scene_create: an invalid one is RT_ERR_INVALID naming the
    description whatever the handle (here none), and so is it for the refit check"""
    sc = rt.Scene.from_file(scene_path("spheres.json"), random_spheres_seed=1)
    d = sc.desc()
    mats = np.ctypeslib.as_array(d.material, shape=(d.n_shapes,)).copy()
    mats[0] = d.n_materials
    d.material = mats.ctypes.data_as(C.POINTER(C.c_uint32))
    core = _ffi.core()
    assert core.rt_scene_update(None, C.byref(d)) == _ffi.RT_ERR_INVALID
    assert b"material index out of range" in core.rt_last_error()
    assert core.rt_scene_update(None, None) == _ffi.RT_ERR_INVALID
    assert b"null scene description" in core.rt_last_error()
    worst = C.c_double()
    assert core.rt_cull_refit_check(C.byref(d), 0, None, None, C.byref(worst)) == _ffi.RT_ERR_INVALID
    good = sc.desc()
    assert core.rt_scene_update(None, C.byref(good)) == _ffi.RT_ERR_INVALID
    assert b"null scene" in core.rt_last_error()


@pytest.mark.skipif(rt.device_count() > 0, reason="checks the behaviour without a CUDA device")
def test_entries_fail_loudly_without_a_device():
    """no handle can exist without a device (rt_scene_create: RT_ERR_NO_DEVICE), so the update entries have nothing to
    run on; a host scene still takes transforms (its description), and asking for its handle afterwards fails"""
    sc = rt.Scene.from_file(scene_path("spheres.json"), random_spheres_seed=1)
    out = C.c_void_p()
    assert _ffi.core().rt_scene_create(C.byref(sc.desc()), 0, C.byref(out)) == _ffi.RT_ERR_NO_DEVICE
    sc.set_transforms([3], [(1.0, 2.0, 3.0)], [(0, 0, 0)], [(0.5, 0.5, 0.5)])
    with pytest.raises(rt.RtError):
        sc.device_scene()


def test_scene_set_transforms_edits_the_description():
    """Scene.set_transforms (rth_scene_set_transforms) gives the rows the JSON loader gives for the same transforms;
    bad and repeated indices are rejected before anything changes"""
    base = dict(TRIO)
    shapes = [{"type": "Sphere", "name": f"s{k}", "material": "M",
               "transform": {"translate": [k, 0, 0], "rotate": [0, 0, 0], "scale": [0.5, 0.5, 0.5]}} for k in range(4)]
    moved = [dict(s) for s in shapes]
    moved[1] = dict(moved[1], transform={"translate": [5, 1, 2], "rotate": [10, 20, 30], "scale": [0.5, 1.0, 2.0]})
    moved[3] = dict(moved[3], transform={"translate": [-1, -2, 0], "rotate": [0, 90, 0], "scale": [2, 2, 2]})
    sc = rt.Scene.from_json(json.dumps(dict(base, shapes=shapes)), add_random_spheres=False)
    want = rt.Scene.from_json(json.dumps(dict(base, shapes=moved)), add_random_spheres=False).desc()
    rows = lambda d, f: np.ctypeslib.as_array(getattr(d, f), shape=(d.n_shapes, 12)).copy()
    before = rows(sc.desc(), "inverse")
    for bad in ([4], [1, 1]):
        with pytest.raises(rt.RtError):
            sc.set_transforms(bad, [(0, 0, 0)] * len(bad), [(0, 0, 0)] * len(bad), [(1, 1, 1)] * len(bad))
    assert np.array_equal(rows(sc.desc(), "inverse"), before)
    sc.set_transforms([3, 1], [(-1, -2, 0), (5, 1, 2)], [(0, 90, 0), (10, 20, 30)], [(2, 2, 2), (0.5, 1.0, 2.0)])
    got = sc.desc()
    for f in ("inverse", "direct"):
        assert np.array_equal(rows(got, f), rows(want, f)), f


def test_translated_rows_and_random_walk():
    """api.translated_rows is translate(shift) o T: the rows of the loader's transform with the translation moved"""
    t = ((0.5, -1.0, 2.0), (10.0, 20.0, 30.0), (0.5, 0.75, 2.0))
    inv, direct = api.transform(*t)
    inv2, direct2 = api.translated_rows(inv[None], direct[None], [(1.0, -2.0, 0.5)])
    want_inv, want_dir = api.transform((1.5, -3.0, 2.5), t[1], t[2])
    assert np.allclose(inv2[0], want_inv, rtol=0, atol=1e-14) and np.allclose(direct2[0], want_dir, rtol=0, atol=1e-14)
    sc = rt.Scene.from_file(scene_path("spheres.json"), random_spheres_seed=1)
    walk = api.random_walk(sc, [7, 9], 3, 0.1, seed=2)
    assert len(walk) == 3 and all(w[0].tolist() == [7, 9] and w[1].shape == (2, 12) for w in walk)
    assert np.array_equal(walk[0][2].reshape(2, 3, 4)[:, 1, 3], current_direct(sc)[[7, 9]].reshape(2, 3, 4)[:, 1, 3])


def current_direct(sc):
    d = sc.desc()
    return np.ctypeslib.as_array(d.direct, shape=(d.n_shapes, 12)).copy()


def test_python_argument_checks():
    good = (np.zeros(2, np.uint32), np.zeros((2, 12)), np.zeros((2, 12)))
    api.check_transforms(*good)
    for bad in ((np.zeros(2, np.int64), good[1], good[2]), (np.zeros((2, 1), np.uint32), good[1], good[2]),
                (good[0], np.zeros((2, 12), np.float32), good[2]), (good[0], good[1], np.zeros((3, 12))),
                (good[0], np.zeros((2, 16)), good[2])):
        with pytest.raises(ValueError):
            api.check_transforms(*bad)
        with pytest.raises(ValueError):
            api.update_transforms(None, *bad)


def test_transform_helper_gives_the_description_rows():
    """api.transform is InversableTransform::new: the rows the JSON loader puts into the description"""
    scene = dict(TRIO)
    t = {"translate": [0.5, -1.25, 2.0], "rotate": [10.0, 20.0, 30.0], "scale": [0.5, 0.75, 2.0]}
    scene["shapes"] = [{"type": "Cube", "name": "c", "material": "M", "transform": t}]
    sc = rt.Scene.from_json(json.dumps(scene), add_random_spheres=False)
    d = sc.desc()
    inv, direct = api.transform(t["translate"], t["rotate"], t["scale"])
    assert np.array_equal(inv, np.ctypeslib.as_array(d.inverse, shape=(12,)))
    assert np.array_equal(direct, np.ctypeslib.as_array(d.direct, shape=(12,)))


@pytest.mark.parametrize("name", FIXTURES)
def test_refit_encloses_after_random_motions_on_fixture_scenes(name):
    sc = rt.Scene.from_file(scene_path(name), random_spheres_seed=1)
    base = current_inverse(sc)
    n = len(base)
    assert refit_worst(sc, [], np.zeros((0, 12))) <= 1e-7
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    for k in (1, 16, n):
        for step in (0.05, 1.0, 20.0):
            index = rng.choice(n, size=min(k, n), replace=False).astype(np.uint32)
            assert refit_worst(sc, index, random_moves(rng, base, index, step)) <= 1e-7, (k, step)


def test_refit_encloses_on_generated_scenes():
    """10^4 shapes: one level above the roots, every kind of node refit"""
    sc = big_scene(10000, seed=5, extent=25.0)
    base = current_inverse(sc)
    n = len(base)
    rng = np.random.default_rng(6)
    for k in (1, 16, n):
        index = rng.choice(n, size=k, replace=False).astype(np.uint32)
        assert refit_worst(sc, index, random_moves(rng, base, index, 3.0)) <= 1e-7, k


def test_refit_encloses_after_100_random_walk_steps():
    """The refit recomputes a dirty node from ALL its members' current balls, so its result depends only on the shapes'
    final rows, not on the order of the steps: 100 steps of a random walk of random subsets are checked through their
    end positions (the GPU suite runs the steps one by one)."""
    sc = rt.Scene.from_file(scene_path("spheres.json"), random_spheres_seed=1)
    base = current_inverse(sc)
    n = len(base)
    rng = np.random.default_rng(7)
    cur = base.copy()
    moved = np.zeros(n, bool)
    for _ in range(100):
        index = rng.choice(n, size=16, replace=False)
        cur[index] = random_moves(rng, cur, index, 0.3)
        moved[index] = True
        all_moved = np.flatnonzero(moved).astype(np.uint32)
        assert refit_worst(sc, all_moved, cur[all_moved]) <= 1e-7


@pytest.mark.parametrize("case", ["far", "shrunk", "ill_conditioned", "singular", "nan"])
def test_refit_extreme_motions_and_back(case):
    """shapes flung 1e6 away, shrunk by 1e-6, made ill-conditioned (kappa > 30: never culled, so every node above them
    is never rejected) or singular, or given NaN rows; then moved back"""
    sc = rt.Scene.from_file(scene_path("spheres.json"), random_spheres_seed=1)
    base = current_inverse(sc)
    d = sc.desc()
    direct = np.ctypeslib.as_array(d.direct, shape=(d.n_shapes, 12))
    kinds = sc.shape_kinds()
    rng = np.random.default_rng(8)
    index = rng.choice(np.flatnonzero(kinds == _ffi.RT_SHAPE_SPHERE)[5:], size=16, replace=False).astype(np.uint32)
    rows = []
    for i in index:
        c = direct[i].reshape(3, 4)[:, 3]
        if case == "far":
            inv, _ = api.transform(c + rng.normal(0, 1e6, 3), (0, 0, 0), (0.2, 0.2, 0.2))
        elif case == "shrunk":
            inv, _ = api.transform(c, (0, 0, 0), (2e-7, 2e-7, 2e-7))
        elif case == "ill_conditioned":
            inv, _ = api.transform(c, (10, 20, 30), (0.2, 0.2, 0.2 * 100))
        elif case == "singular":
            inv, _ = api.transform(c, (0, 0, 0), (0.2, 0.0, 0.2))
        else:
            inv = np.full(12, np.nan)
        rows.append(inv)
    assert refit_worst(sc, index, np.array(rows)) <= 1e-7
    assert refit_worst(sc, index, base[index]) <= 1e-7
