"""rt_trace_pixel_samples_group[_device] on the rays callers bring, against the oracle at float precision.

A frame only ever traces camera rays from the camera position, and for those the group entry is pinned bit for bit to
the frame (test_gpu_trace_group.py).  Callers also bring rays that start inside a solid, inside a marched shape's bound,
on a surface or far away; axis-aligned directions with signed zeros; directions that are not of unit length (the ABI
takes them as given: neither the library nor the oracle normalises); NaN and Inf rays; and the pixel key 0xFFFFFFFF,
which no frame can use.

The strict comparison (check_groups) is check_pixels' bound applied group by group: the oracle's per-ray FP64 colours
(group_sample_colors) are rounded to float, summed in f64 in ray order from 0.0 and divided by the group's count, and
each path may be off by one float ulp.  The number of groups not bit-identical to that emulated mean is printed."""
import numpy as np
import pytest

import rs_pathtracing_b200 as rt
from oracle import pyoracle as po

from conftest import scene_path
from test_gpu_frame_edges import SEEDS
from test_gpu_trace_group import _variant_4b

pytestmark = pytest.mark.gpu

DEPTH = 8


def _emulated(cols, offsets):
    """(f32 colours, f64 in-order group sums, counts) of the oracle's per-ray colours"""
    f32 = np.asarray(cols, dtype=np.float64).astype(np.float32)
    f = f32.astype(np.float64)
    off = np.asarray(offsets, dtype=np.int64)
    n = np.diff(off)
    s = np.zeros((len(n), 3))
    for k in range(int(n.max(initial=0))):
        m = n > k
        s[m] = s[m] + f[off[:-1][m] + k]
    return f32, s, n


def check_groups(got, cols, offsets, what=""):
    """got: GPU group means (G, 3); cols: the oracle's per-ray colours (n_rays, 3) in ray order; offsets: G + 1 group
    starts.  Asserts check_pixels' bound group by group; returns the number of groups not bit-identical to the emulated
    mean.  An empty group must be NaN in all three channels; a channel whose emulated mean is not finite must be NaN
    where it is NaN and the same infinity where it is infinite."""
    got = np.asarray(got, dtype=np.float64).reshape(-1, 3)
    f32, s, n = _emulated(cols, offsets)
    assert got.shape[0] == len(n), (got.shape, len(n))
    off = np.asarray(offsets, dtype=np.int64)
    with np.errstate(invalid="ignore", divide="ignore"):
        emu = s / n[:, None]
    empty = n == 0
    assert np.isnan(got[empty]).all(), f"{what}: an empty group is not NaN"
    # per group: the sum of the float ulps of its paths (non-finite paths give NaN here: those channels are not finite)
    ulps = np.zeros((len(n), 3))
    with np.errstate(invalid="ignore"):
        sp = np.spacing(np.abs(f32)).astype(np.float64)
        for k in range(int(n.max(initial=0))):
            m = n > k
            ulps[m] = ulps[m] + sp[off[:-1][m] + k]
        bound = ulps / np.maximum(n, 1)[:, None] + n[:, None] * np.spacing(np.abs(emu))
    one = n == 1
    f0 = np.zeros((len(n), 3), np.float32)
    f0[one] = f32[off[:-1][one]]
    lo = np.nextafter(f0, np.float32(-np.inf)).astype(np.float64)
    hi = np.nextafter(f0, np.float32(np.inf)).astype(np.float64)
    finite = np.isfinite(emu)
    with np.errstate(invalid="ignore"):
        ok = np.where(one[:, None], (got == emu) | (got == lo) | (got == hi), np.abs(got - emu) <= bound)
    ok = np.where(finite, ok, (np.isnan(emu) & np.isnan(got)) | (np.isinf(emu) & (got == emu)))
    bad = ~ok.all(axis=1) & ~empty
    if bad.any():
        i = int(np.flatnonzero(bad)[0])
        raise AssertionError(f"{what}: {int(bad.sum())} of {len(n)} groups exceed one float ulp per path; first: group {i} "
                             f"of {int(n[i])} rays, gpu {got[i].tolist()}, emulated {emu[i].tolist()}, "
                             f"bound {bound[i].tolist()}")
    same = ((got == emu) | (np.isnan(got) & np.isnan(emu))).all(axis=1)
    n_diff = int((~same & ~empty).sum())
    print(f"strict-bound {what}: {n_diff} of {int((~empty).sum())} groups not bit-identical")
    return n_diff


# ---- caller rays -------------------------------------------------------------------------------------------------

def _load(name, variant=""):
    sc = rt.Scene.from_file(scene_path(name), random_spheres_seed=1)
    cam = _variant_4b(sc) if variant == "4b" else sc.camera()
    return sc, cam


def _centre(sc, i):
    """the origin of shape i's local frame in world space: inside a sphere or cube, the centre of a marched shape's
    bounding ball"""
    d = sc.desc()
    m = np.ctypeslib.as_array(d.direct, shape=(d.n_shapes, 12))[i]
    return m[[3, 7, 11]].copy()


def _unit(rng, n):
    d = rng.normal(size=(n, 3))
    return d / np.linalg.norm(d, axis=1, keepdims=True)


def _axes():
    """the six axis-aligned unit directions, each with its other two components +0/+0, -0/-0 and +0/-0"""
    out = []
    for a in range(3):
        for sign in (1.0, -1.0):
            for zeros in ((0.0, 0.0), (-0.0, -0.0), (0.0, -0.0)):
                d = [zeros[0], zeros[1]]
                d.insert(a, sign)
                out.append(d)
    return np.array(out)


AXES = _axes()


def _ray_sets(sc, cam, inside, rng):
    """named (n, 6) ray sets: origins inside the shapes `inside`, on surface points the oracle's intersection returns,
    1e5 units away aimed at the scene, at the camera with axis-aligned signed-zero directions, and directions of length
    0.5 and 3"""
    pos = np.array(cam.position.tuple())
    aim = np.array(cam.direction.tuple())
    sets = {}
    for i in inside:
        c = _centre(sc, i)
        o = np.concatenate([c[None], c + 0.05 * _unit(rng, 7)])
        sets[f"inside shape {i}"] = np.concatenate([np.repeat(o, 4, axis=0), _unit(rng, 32)], axis=1)
        sets[f"inside shape {i}, axes"] = np.concatenate([np.tile(c, (len(AXES), 1)), AXES], axis=1)
    probe = np.concatenate([np.tile(pos, (256, 1)), _unit(rng, 256) * 0.3 + aim], axis=1)
    probe[:, 3:] /= np.linalg.norm(probe[:, 3:], axis=1, keepdims=True)
    hit = po.OracleScene(sc.desc()).intersect_batch(probe)
    pts = hit["point"][hit["index"] >= 0][:33]
    assert len(pts) >= 17
    sets["on a surface"] = np.concatenate([pts, _unit(rng, len(pts))], axis=1)
    far = _unit(rng, 17)
    target = pos + 10.0 * aim
    sets["1e5 away"] = np.concatenate([target + 1e5 * far, -far], axis=1)
    sets["camera, axes"] = np.concatenate([np.tile(pos, (len(AXES), 1)), AXES], axis=1)
    for length in (0.5, 3.0):
        d = (_unit(rng, 31) * 0.2 + aim)
        d = length * d / np.linalg.norm(d, axis=1, keepdims=True)
        sets[f"length {length}"] = np.concatenate([np.tile(pos, (31, 1)), d], axis=1)
    return sets


def _grouped(sets, sizes, pix_pool, rng):
    """the ray sets cut into consecutive groups of the given sizes (cycled), with pixel indices drawn from pix_pool"""
    rays = np.concatenate(list(sets.values())).reshape(-1, 6)
    sizes_out, r = [], 0
    k = 0
    while r < len(rays):
        n = min(sizes[k % len(sizes)], len(rays) - r)
        sizes_out.append(n)
        r += n
        k += 1
    offsets = np.concatenate([[0], np.cumsum(sizes_out)]).astype(np.uint64)
    pix = rng.choice(np.asarray(pix_pool, np.uint32), len(sizes_out)).astype(np.uint32)
    pix[0], pix[-1] = pix_pool[0], pix_pool[1]
    return rays, offsets, pix


GROUP_SIZES = [1, 15, 0, 16, 17, 31, 0, 0, 32, 33]
PIX_POOL = [0, 0xFFFFFFFF, 0xFFFFFFFE, 7, 7, 123456]

# (scene, variant, shapes to start inside: a Dielectric sphere, a Cube, marched shapes' bounding balls)
CASES = [("spheres.json", "", [1, 2, 3], SEEDS[1]),             # glass spheres (outer, inner), marched Sphere2
         ("cornell_box.json", "", [6, 8], SEEDS[2]),            # Cube1, the heart
         ("dupin.json", "", [0], SEEDS[3]),                     # the cyclide
         ("detached_materials.json", "4b", [1, 2], SEEDS[4])]   # EarthMap metal sphere, glass Hunt's surface


@pytest.mark.parametrize("name,variant,inside,seed", CASES)
def test_caller_rays_match_oracle(name, variant, inside, seed):
    """every kind of caller ray in groups of 1 to 33 rays, empty groups among them, keys 0 and 0xFFFFFFFF and repeated
    keys: the strict bound against the oracle's per-ray colours; the _device form on a torch side stream gives the host
    form's means bit for bit"""
    sc, cam = _load(name, variant)
    osc = po.OracleScene(sc.desc())
    rng = np.random.default_rng(17)
    rays, offsets, pix = _grouped(_ray_sets(sc, cam, inside, rng), GROUP_SIZES, PIX_POOL, rng)
    assert {0, 0xFFFFFFFF} <= set(pix.tolist())
    got = sc.trace_pixel_samples_group(rays, offsets, pix, DEPTH, seed=seed)
    cols = osc.group_sample_colors(rays, offsets, pix, DEPTH, seed)
    check_groups(got, cols, offsets, f"{name}{variant} caller rays")
    torch = pytest.importorskip("torch")
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        t = torch.from_numpy(rays).to("cuda", non_blocking=True)
        dev = sc.trace_pixel_samples_group(t, offsets, pix, DEPTH, seed=seed).cpu().numpy()
    s.synchronize()
    assert np.array_equal(dev, got, equal_nan=True)


@pytest.mark.parametrize("seed", SEEDS)
def test_caller_ray_seeds(seed):
    """both words of the RNG key on caller rays with the keys 0 and 0xFFFFFFFF"""
    sc, cam = _load("spheres.json")
    rng = np.random.default_rng(seed % 1000)
    sets = _ray_sets(sc, cam, [1], rng)
    rays, offsets, pix = _grouped(sets, [3, 1, 8, 0], [0, 0xFFFFFFFF, 99], rng)
    got = sc.trace_pixel_samples_group(rays, offsets, pix, DEPTH, seed=seed)
    check_groups(got, po.OracleScene(sc.desc()).group_sample_colors(rays, offsets, pix, DEPTH, seed), offsets,
                 f"seed {seed}")


@pytest.mark.parametrize("name", ["spheres.json", "cornell_box.json"])
def test_non_finite_rays(name):
    """one NaN ray and one Inf ray, each in an otherwise normal group: those groups have the oracle's non-finite means,
    and every other group is what it is without them, bit for bit"""
    sc, cam = _load(name)
    osc = po.OracleScene(sc.desc())
    rng = np.random.default_rng(5)
    pos = np.array(cam.position.tuple())
    aim = np.array(cam.direction.tuple())
    d = _unit(rng, 40) * 0.2 + aim
    good = np.concatenate([np.tile(pos, (40, 1)), d / np.linalg.norm(d, axis=1, keepdims=True)], axis=1)
    bad_rays = {"nan direction": np.r_[pos, np.nan, 0.0, 1.0], "nan origin": np.r_[np.nan, pos[1:], aim],
                "inf direction": np.r_[pos, 0.0, np.inf, 0.0], "inf origin": np.r_[-np.inf, pos[1:], aim],
                "inf everywhere": np.r_[np.inf, np.inf, np.inf, -np.inf, np.inf, np.inf]}
    for what, bad in bad_rays.items():
        # groups of 10: the bad ray is ray 4 of group 1
        rays = np.concatenate([good[:14], bad[None], good[14:]])
        offsets = np.array([0, 10, 21, 31, 41], np.uint64)
        pix = np.array([3, 4, 5, 6], np.uint32)
        got = sc.trace_pixel_samples_group(rays, offsets, pix, DEPTH, seed=11)
        cols = osc.group_sample_colors(rays, offsets, pix, DEPTH, 11)
        check_groups(got, cols, offsets, f"{name} {what}")
        ref = sc.trace_pixel_samples_group(good, np.array([0, 10, 20, 30, 40], np.uint64), pix, DEPTH, seed=11)
        assert np.array_equal(got[[0, 2, 3]], ref[[0, 2, 3]]), what


def _batch_groups(cap):
    """groups around RT_B200_BATCH_PATHS = cap: exactly one batch, one batch plus one ray, two batches plus one ray,
    with empty groups first, last, and right before and after the split groups"""
    return [0, 3, cap, 0, cap + 1, 0, 1, 0, 2 * cap + 1, 0, 5, 16, 17, 0, cap - 1, 2, 0]


@pytest.mark.parametrize("lanes", [1, 3])
def test_groups_around_batch_boundaries(monkeypatch, lanes):
    cap = 40
    name = "cornell_box.json"
    sc, cam = _load(name)
    osc = po.OracleScene(sc.desc())
    rng = np.random.default_rng(9)
    sets = _ray_sets(sc, cam, [6, 8], rng)
    pool = np.concatenate(list(sets.values()))
    sizes = _batch_groups(cap)
    rays = pool[rng.integers(0, len(pool), sum(sizes))]
    offsets = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    pix = rng.choice(np.array(PIX_POOL, np.uint32), len(sizes)).astype(np.uint32)
    seed = SEEDS[3]
    ref = sc.trace_pixel_samples_group(rays, offsets, pix, DEPTH, seed=seed)
    check_groups(ref, osc.group_sample_colors(rays, offsets, pix, DEPTH, seed), offsets, f"batch groups, {lanes} lanes")
    monkeypatch.setenv("RT_B200_BATCH_PATHS", str(cap))
    monkeypatch.setenv("RT_B200_LANES", str(lanes))
    small, _ = _load(name)   # a new device handle reads the variables
    assert np.array_equal(small.trace_pixel_samples_group(rays, offsets, pix, DEPTH, seed=seed), ref, equal_nan=True)
    torch = pytest.importorskip("torch")
    dev = small.trace_pixel_samples_group(torch.from_numpy(rays).cuda(), offsets, pix, DEPTH, seed=seed)
    assert np.array_equal(dev.cpu().numpy(), ref, equal_nan=True)


def test_many_small_groups():
    """10^5 groups of 1 to 3 rays in one call (the loader's binary search over the whole offset table), keys spread
    over the 32-bit range"""
    sc, cam = _load("spheres.json")
    rng = np.random.default_rng(21)
    sizes = rng.integers(1, 4, 100_000)
    n = int(sizes.sum())
    pos = np.array(cam.position.tuple())
    aim = np.array(cam.direction.tuple())
    d = _unit(rng, n) * 0.4 + aim
    rays = np.concatenate([np.tile(pos, (n, 1)), d / np.linalg.norm(d, axis=1, keepdims=True)], axis=1)
    offsets = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    pix = rng.integers(0, 1 << 32, len(sizes), dtype=np.uint64).astype(np.uint32)
    pix[:2] = [0, 0xFFFFFFFF]
    depth, seed = 4, SEEDS[2]
    got = sc.trace_pixel_samples_group(rays, offsets, pix, depth, seed=seed)
    check_groups(got, po.OracleScene(sc.desc()).group_sample_colors(rays, offsets, pix, depth, seed), offsets,
                 "1e5 small groups")
