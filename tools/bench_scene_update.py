"""Scene updates on a live handle against a new handle, on one GPU:

  python tools/bench_scene_update.py [--out profiles/scene_update_bench_1gpu.json] [--reps 5] [--frames 20]

  1. rt_scene_update (a whole new description in place) against rt_scene_destroy + rt_scene_create, each followed by
     the first frame (640x480x1, depth 8): spheres, cornell_box and generated scenes of 10^4 and 10^5 shapes
     (tests/test_cull_cpu.py:big_scene);
  2. per-frame time of an animation moving 1, 16 and all 481 random spheres on a seeded random walk, at spheres
     640x480x1 spp and cornell_box 1600x900x1 spp (depth 50, the bins' setting): rt_scene_update_transforms + frame on
     one handle against a new handle of the edited description per frame (create + frame + destroy);
  3. tree degradation after 100 random-walk refits of every random sphere: k_extend device time of one frame (kernel
     timing on) and FAST Mrays/s of rt_intersect_batch on 2^20 rays, refit handle against a handle rebuilt from the
     same description; every frame of the comparison is checked equal.
Host clock around work that ends in a device synchronise; medians of --reps.  The card's name and power limit are read
in the same run.  Needs a CUDA device."""
import argparse, ctypes as C, json, os, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import rs_pathtracing_b200 as rt
from rs_pathtracing_b200 import _ffi, api

ap = argparse.ArgumentParser()
ap.add_argument("--out", default=None)
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--frames", type=int, default=20)
a = ap.parse_args()
if rt.device_count() == 0:
    sys.exit("bench_scene_update needs a CUDA device")
core = _ffi.core()


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        return q
    except Exception as e:   # the numbers stay, the card is then unknown
        return f"unknown ({e})"


def create(desc):
    h = C.c_void_p()
    api._check(core.rt_scene_create(C.byref(desc), 0, C.byref(h)))
    return h


def frame(h, cam, w, hh, spp, depth, seed=1):
    api.render_start(h, cam, api.render_params(w, hh, spp, depth, seed))
    buf = np.empty((hh, w, 3))
    api.render_wait(h, buf)
    return buf


def med(xs):
    return float(np.median(xs))


class Rows:
    """a scene's description with editable inverse / direct rows"""

    def __init__(self, sc):
        self.sc = sc
        d = sc.desc()
        self.inv = np.ctypeslib.as_array(d.inverse, shape=(d.n_shapes, 12)).copy()
        self.dir = np.ctypeslib.as_array(d.direct, shape=(d.n_shapes, 12)).copy()

    def desc(self):
        d = self.sc.desc()
        d.inverse = self.inv.ctypes.data_as(C.POINTER(C.c_double))
        d.direct = self.dir.ctypes.data_as(C.POINTER(C.c_double))
        return d


def load(name):
    if name.startswith("big"):
        from test_cull_cpu import big_scene
        n = int(float(name[3:]))
        return big_scene(n, seed=3, extent=30.0 * (n / 2e4) ** (1 / 3))
    return rt.Scene.from_file(os.path.join(ROOT, "scenes", name), random_spheres_seed=1)


out = {"card": card(), "full_update": [], "animation": [], "degradation": []}
spheres_cam = load("spheres.json").camera()

# 1. full update against a new handle
for name in ("spheres.json", "cornell_box.json", "big1e4", "big1e5"):
    sc = load(name)
    cam = sc.camera() if not name.startswith("big") else rt.camera_new((0, 5, -60), (0, -0.05, 1), (0, 1, 0), 1.0, 0.8)
    other = load("cornell_box.json" if name != "cornell_box.json" else "spheres.json")
    h = create(sc.desc())
    frame(h, cam, 640, 480, 1, 8)
    upd, new = [], []
    for _ in range(a.reps):
        api.scene_update(h, other.desc())
        t0 = time.perf_counter()
        api.scene_update(h, sc.desc())
        f_upd = frame(h, cam, 640, 480, 1, 8)
        upd.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        g = create(sc.desc())
        f_new = frame(g, cam, 640, 480, 1, 8)
        core.rt_scene_destroy(g)
        new.append(time.perf_counter() - t0)
        assert np.array_equal(f_upd, f_new), name
    core.rt_scene_destroy(h)
    row = {"scene": name, "shapes": sc.shape_count, "update_plus_frame_ms": med(upd) * 1e3,
           "create_plus_frame_ms": med(new) * 1e3}
    out["full_update"].append(row)
    print(json.dumps(row), flush=True)

# 2. animation: refit + frame on one handle against a new handle per frame
for name, (w, hh) in (("spheres.json", (640, 480)), ("cornell_box.json", (1600, 900))):
    sc = load(name)
    cam = sc.camera()
    n_file = rt.Scene.from_file(os.path.join(ROOT, "scenes", name), add_random_spheres=False).shape_count
    randoms = np.arange(n_file, sc.shape_count)
    for k in (1, 16, len(randoms)):
        walk = api.random_walk(sc, randoms[:k], a.frames, 0.05, seed=k)
        rows = Rows(sc)
        h = create(rows.desc())
        frame(h, cam, w, hh, 1, 50)
        t_upd, t_new, t_refit = [], [], []
        for index, inv, direct in walk:
            t0 = time.perf_counter()
            api.update_transforms(h, index, inv, direct)
            t_refit.append(time.perf_counter() - t0)
            f_upd = frame(h, cam, w, hh, 1, 50)
            t_upd.append(time.perf_counter() - t0)
            rows.inv[index], rows.dir[index] = inv, direct
            t0 = time.perf_counter()
            g = create(rows.desc())
            f_new = frame(g, cam, w, hh, 1, 50)
            core.rt_scene_destroy(g)
            t_new.append(time.perf_counter() - t0)
            assert np.array_equal(f_upd, f_new), (name, k)
        core.rt_scene_destroy(h)
        row = {"scene": name, "size": [w, hh, 1], "moving": int(k), "frames": a.frames,
               "update_transforms_call_ms": med(t_refit) * 1e3, "update_plus_frame_ms": med(t_upd) * 1e3,
               "new_handle_plus_frame_ms": med(t_new) * 1e3}
        out["animation"].append(row)
        print(json.dumps(row), flush=True)

# 3. tree degradation after 100 refits
for name in ("spheres.json", "big1e4"):
    sc = load(name)
    cam = sc.camera() if not name.startswith("big") else rt.camera_new((0, 5, -60), (0, -0.05, 1), (0, 1, 0), 1.0, 0.8)
    n_file = (rt.Scene.from_file(os.path.join(ROOT, "scenes", name), add_random_spheres=False).shape_count
              if not name.startswith("big") else 0)
    movers = np.flatnonzero(sc.shape_kinds() == _ffi.RT_SHAPE_SPHERE)
    movers = movers[movers >= n_file][:20000]
    rows = Rows(sc)
    h = create(rows.desc())
    step = 0.05 if not name.startswith("big") else 0.3
    for index, inv, direct in api.random_walk(sc, movers, 100, step, seed=7):
        api.update_transforms(h, index, inv, direct)
        rows.inv[index], rows.dir[index] = inv, direct
    g = create(rows.desc())
    rng = np.random.default_rng(1)
    o = rng.uniform(-20, 20, (1 << 20, 3)) + (0, 10, 0)
    rays = rt.make_rays(o, rng.uniform(-10, 10, (1 << 20, 3)) - o)
    idx = np.empty(len(rays), np.int32)
    res = {}
    for label, hd in (("refit", h), ("rebuilt", g)):
        core.rt_set_kernel_timing(hd, 1)
        ext, rate = [], []
        for _ in range(a.reps):
            core.rt_reset_stats(hd)
            f = frame(hd, cam, 640, 480, 1, 8)
            st = rt.Stats()
            core.rt_get_stats(hd, C.byref(st))
            ext.append(st.ms_extend)
            api._check(core.rt_intersect_batch(hd, rays.ctypes.data_as(C.c_void_p), len(rays), 0.001, np.inf,
                                               rt.RT_ISECT_FAST, idx.ctypes.data_as(C.c_void_p), None, None, None,
                                               None, None))
            core.rt_get_stats(hd, C.byref(st))
            rate.append(len(rays) / (st.last_intersect_ms * 1e-3) / 1e6)
        core.rt_set_kernel_timing(hd, 0)
        res[label] = (f, idx.copy(), med(ext), med(rate))
    assert np.array_equal(res["refit"][0], res["rebuilt"][0]) and np.array_equal(res["refit"][1], res["rebuilt"][1])
    core.rt_scene_destroy(h)
    core.rt_scene_destroy(g)
    row = {"scene": name, "moving": int(len(movers)), "refits": 100, "step": step,
           "k_extend_ms_refit": res["refit"][2], "k_extend_ms_rebuilt": res["rebuilt"][2],
           "fast_mrays_refit": res["refit"][3], "fast_mrays_rebuilt": res["rebuilt"][3]}
    out["degradation"].append(row)
    print(json.dumps(row), flush=True)

print(json.dumps({"card": out["card"]}))
if a.out:
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
