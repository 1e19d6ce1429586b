#!/usr/bin/env python
"""Occlusion queries (rt_occluded_batch_device, RT_ISECT_FAST) against the nearest hit (rt_intersect_batch_device,
RT_ISECT_FAST, shape index only) on the same device-resident rays.

  python tools/bench_occluded.py [--warmup 2] [--reps 10] [--out profiles/occluded_bench_1gpu.json]

Prints one JSON line per ray set and one summary line (written to --out when given).  Needs a CUDA device; reads the
GPU's name and power limit with a read-only nvidia-smi query in the same run.  Times are CUDA events around each launch
on one stream (torch's current stream), medians over --reps with the two queries alternated rep by rep.  The nearest
hit gets the same per-ray bound as a scalar when the set has one, and +inf otherwise (it has no per-ray bound).

Ray sets:
  (a) bench.py config 2's 1 Mi rays: the bench trio (Sphere, Cube, Heart) with test_gpu_intersect.bench_rays, and the
      cornell_box shape list with test_gpu_intersect.scene_rays; t_max = inf.
  (b) shadow rays: the hit points of cornell_box's 1024x1024 camera rays (one jittered sample each) toward uniform points of its
      ceiling light, t_max = (1 - 1e-9) * distance.
  (c) the same on dupin (a ray-marched Dupin cyclide); dupin has no emitter, so the targets are uniform points of a
      6 x 6 square 8 units above the origin.
  (d) a generated 10^4-shape scene (tools/big_scene_probe.py's generator, levels above the roots): 1 Mi box rays with
      t_max = inf, and the same rays as segments to their targets.
Per set: Mrays/s of both queries, the occluded fraction, and shape tests / cull tests / march evaluations per ray from
the counters (a separate host-form run with counters on).  Both queries' answers are checked against each other.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

import rs_pathtracing_b200 as rt  # noqa: E402
from rs_pathtracing_b200 import _ffi, api  # noqa: E402
from bench_adaptive import gpu_info  # noqa: E402
from bench_trace_group import camera_rays  # noqa: E402
from test_cull_cpu import big_scene, box_rays  # noqa: E402
from test_gpu_intersect import TRIO, bench_rays, scene_rays  # noqa: E402

N = 1 << 20


def load(name):
    return rt.Scene.from_file(os.path.join(ROOT, "scenes", name), random_spheres_seed=1)


def shadow_set(sc, targets_fn, rng):
    """hit points of 1024^2 jittered camera rays toward targets_fn(n) points"""
    cam = sc.camera()
    rays = camera_rays(cam, 1024, 1024, 1, rng)
    hits = sc.closest_hit(rays, mode=rt.RT_ISECT_FAST, want=("index", "point"))
    pts = hits["point"][hits["index"] >= 0]
    srays, dist = api.shadow_rays(pts, targets_fn(len(pts)))
    ok = dist > 0
    return srays[ok], np.ascontiguousarray((1 - 1e-9) * dist[ok])


def cornell_light(sc, rng):
    d = sc.desc()
    i = next(i for i in range(d.n_shapes) if d.materials[d.material[i]].kind == _ffi.RT_MAT_DIFFUSE_LIGHT)
    q = np.ctypeslib.as_array(d.params, shape=(d.n_shapes, 8))[i]
    m = np.ctypeslib.as_array(d.direct, shape=(d.n_shapes, 12))[i].reshape(3, 4)

    def targets(n):
        u = rng.uniform(0, 1, (n, 2))
        obj = np.stack([q[0] + u[:, 0] * (q[2] - q[0]), q[1] + u[:, 1] * (q[3] - q[1]), np.zeros(n)], 1)
        return obj @ m[:, :3].T + m[:, 3]
    return targets


def square_above(rng):
    def targets(n):
        u = rng.uniform(-3.0, 3.0, (n, 2))
        return np.stack([u[:, 0], np.full(n, 8.0), u[:, 1]], 1)
    return targets


def ray_sets():
    rng = np.random.default_rng(2024)
    trio = rt.Scene.from_json(json.dumps(TRIO), add_random_spheres=False)
    cornell = load("cornell_box.json")
    dupin = load("dupin.json")
    big = big_scene(10000, seed=5, extent=25.0)
    o = rng.uniform(-37.5, 37.5, (N, 3))
    tgt = rng.uniform(-25.0, 25.0, (N, 3))
    seg, seg_len = api.shadow_rays(o, tgt)
    yield "a_cfg2_trio", trio, bench_rays(N), math.inf
    yield "a_cfg2_cornell", cornell, scene_rays(cornell, N, seed=9), math.inf
    yield "b_shadow_cornell", cornell, *shadow_set(cornell, cornell_light(cornell, rng), rng)
    yield "c_shadow_dupin", dupin, *shadow_set(dupin, square_above(rng), rng)
    yield "d_big_10k_inf", big, box_rays(N, seed=7, extent=25.0), math.inf
    yield "d_big_10k_segments", big, seg, np.ascontiguousarray((1 - 1e-9) * seg_len)


def per_ray_work(sc, fn, n):
    sc.set_counters(True)
    sc.reset_stats()
    fn()
    st = sc.stats()
    sc.set_counters(False)
    return {"shape_tests": st.shape_tests / n, "cull_tests": st.cull_tests / n, "march_evals": st.march_steps / n,
            "march_rays": st.march_rays / n}


def run_set(name, sc, rays, t_max, warmup, reps):
    import torch
    rays = np.ascontiguousarray(rays, np.float64)
    n = len(rays)
    h = sc.device_scene(0)
    d_rays = torch.from_numpy(rays).cuda()
    per_ray = not np.isscalar(t_max)
    d_tmax = torch.from_numpy(t_max).cuda() if per_ray else float(t_max)
    isect_tmax = math.inf if per_ray else float(t_max)
    occ = torch.empty(n, dtype=torch.uint8, device="cuda")
    idx = torch.empty(n, dtype=torch.int32, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream or 1
    core = _ffi.core()

    def occluded():
        api.occluded_device(h, d_rays, occ, t_max=d_tmax, mode=rt.RT_ISECT_FAST)

    def nearest():
        api._check(core.rt_intersect_batch_device(h, d_rays.data_ptr(), n, 0.001, isect_tmax, rt.RT_ISECT_FAST,
                                                  idx.data_ptr(), None, None, None, None, None, stream))

    fns = {"occluded": occluded, "nearest": nearest}
    for fn in fns.values():
        for _ in range(warmup):
            fn()
    ms = {k: [] for k in fns}
    for _ in range(reps):
        for k, fn in fns.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            ms[k].append(a.elapsed_time(b))
    ms = {k: float(np.median(v)) for k, v in ms.items()}
    got = occ.cpu().numpy().astype(bool)
    # the answers: occluded == the nearest hit's index != -1 (with a scalar bound; per-ray bounds against the literal
    # any-hit loop, RT_ISECT_BRUTE)
    if not per_ray:
        want = sc.closest_hit(rays, 0.001, isect_tmax, mode=rt.RT_ISECT_FAST, want=("index",))["index"] >= 0
        assert np.array_equal(got, want), f"{name}: occluded differs from the nearest hit"
    else:
        assert np.array_equal(got, sc.occluded(rays, 0.001, t_max, mode=rt.RT_ISECT_BRUTE)), name
    row = {"set": name, "rays": n, "t_max": "per ray" if per_ray else str(t_max), "occluded_fraction": float(got.mean()),
           "occluded_ms": ms["occluded"], "nearest_ms": ms["nearest"],
           "occluded_mrays_s": n / ms["occluded"] / 1e3, "nearest_mrays_s": n / ms["nearest"] / 1e3,
           "speedup": ms["nearest"] / ms["occluded"],
           "occluded_work_per_ray": per_ray_work(sc, lambda: sc.occluded(rays, 0.001, t_max), n),
           "nearest_work_per_ray": per_ray_work(sc, lambda: sc.closest_hit(rays, 0.001, isect_tmax, mode=rt.RT_ISECT_FAST,
                                                                           want=("index",)), n)}
    return row


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if rt.device_count() == 0:
        raise SystemExit("bench_occluded needs a CUDA device")
    res = {"bench": "occluded", **gpu_info(0), "warmup": args.warmup, "reps": args.reps, "sets": []}
    for name, sc, rays, t_max in ray_sets():
        row = run_set(name, sc, rays, t_max, args.warmup, args.reps)
        print(json.dumps(row), flush=True)
        res["sets"].append(row)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
