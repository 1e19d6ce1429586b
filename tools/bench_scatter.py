#!/usr/bin/env python
"""What the programmable path costs against the wavefront: rt_scatter_batch_device (RT_ISECT_FAST) against
rt_intersect_batch_device (RT_ISECT_FAST, shape index and t) on the same device-resident rays, and api.trace_paths on
torch against rt_trace_pixel_samples_group_device on the same camera rays.

  python tools/bench_scatter.py [--warmup 2] [--reps 10] [--out profiles/scatter_bench_1gpu.json]

Prints one JSON line per measurement and one summary line (written to --out when given).  Needs a CUDA device; reads the
GPU's name and power limit with a read-only nvidia-smi query in the same run.  Times are CUDA events on torch's current
stream, medians over --reps with the two sides alternated rep by rep.

  (a) rays/s, scatter against nearest hit, on cornell_box, dupin and config 4b (detached_materials with every material
      and texture kind live): the camera rays of a 2048x2048 image (one jittered sample per pixel, 4 Mi rays), and the
      first-bounce rays those of them that scatter leave with (the `scattered` output of level 0).
  (b) paths/s at depth 50 on the camera rays of a 1024x1024 image (1 Mi paths, one per pixel): api.trace_paths on
      torch tensors (one rt_scatter_batch_device per level on the live paths, the throughput and the compaction in torch)
      against the wavefront entry rt_trace_pixel_samples_group_device with one ray per group.  The two results are
      checked bit for bit (api.group_means of the per-ray radiance against the group means) in the same run.
"""
from __future__ import annotations

import argparse
import json
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
from test_gpu_render import _variant_4b  # noqa: E402

DEPTH = 50


def load(name):
    sc = rt.Scene.from_file(os.path.join(ROOT, "scenes", "detached_materials.json" if name == "4b" else name),
                            random_spheres_seed=1)
    return sc, (_variant_4b(sc) if name == "4b" else sc.camera())


def timed(fns, warmup, reps):
    """median ms of each callable, alternated rep by rep"""
    import torch
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
    return {k: float(np.median(v)) for k, v in ms.items()}


def keys_for(n):
    """pixel i, sample 0"""
    return np.ascontiguousarray(np.stack([np.arange(n, dtype=np.uint32), np.zeros(n, np.uint32)], 1))


def scatter_vs_nearest(what, sc, rays, warmup, reps):
    import torch
    rays = np.ascontiguousarray(rays, np.float64)
    n = len(rays)
    h = sc.device_scene(0)
    d_rays = torch.from_numpy(rays).cuda()
    d_keys = torch.from_numpy(keys_for(n).view(np.int32)).cuda()
    new = lambda shape, dt: torch.empty(shape, dtype=dt, device="cuda")
    out = {"index": new((n,), torch.int32), "t": new((n,), torch.float64), "outcome": new((n,), torch.uint8),
           "color": new((n, 3), torch.float64), "scattered": new((n, 6), torch.float64)}
    idx, t = new((n,), torch.int32), new((n,), torch.float64)
    stream = torch.cuda.current_stream().cuda_stream or 1
    core = _ffi.core()

    def scatter():
        api._check(core.rt_scatter_batch_device(h, d_rays.data_ptr(), d_keys.data_ptr(), n, 0, 0, 0.001, np.inf,
                                                rt.RT_ISECT_FAST, *(out[k].data_ptr() for k in api.SCATTER_OUTPUTS),
                                                stream))

    def nearest():
        api._check(core.rt_intersect_batch_device(h, d_rays.data_ptr(), n, 0.001, np.inf, rt.RT_ISECT_FAST,
                                                  idx.data_ptr(), t.data_ptr(), None, None, None, None, stream))

    ms = timed({"scatter": scatter, "nearest": nearest}, warmup, reps)
    assert torch.equal(out["index"], idx) and torch.equal(out["t"].view(torch.int64), t.view(torch.int64)), what
    oc = out["outcome"].cpu().numpy()
    row = {"set": what, "rays": n, "scatter_ms": ms["scatter"], "nearest_ms": ms["nearest"],
           "scatter_mrays_s": n / ms["scatter"] / 1e3, "nearest_mrays_s": n / ms["nearest"] / 1e3,
           "shading_share": 1.0 - ms["nearest"] / ms["scatter"],
           "outcome_fraction": {k: float((oc == v).mean()) for k, v in
                                (("miss", rt.RT_BOUNCE_MISS), ("scatter", rt.RT_BOUNCE_SCATTER), ("emit", rt.RT_BOUNCE_EMIT))}}
    go = np.flatnonzero(oc == rt.RT_BOUNCE_SCATTER)
    return row, out["scattered"][torch.from_numpy(go).cuda()].cpu().numpy()


def paths(what, sc, cam, warmup, reps, seed=7):
    import torch
    w = h = 1024
    rays = np.ascontiguousarray(camera_rays(cam, w, h, 1, np.random.default_rng(3)))
    n = len(rays)
    keys = keys_for(n)
    d_rays = torch.from_numpy(rays).cuda()
    d_keys = torch.from_numpy(keys.view(np.int32)).cuda().view(torch.uint32)
    offsets = np.arange(n + 1, dtype=np.uint64)
    pix = np.arange(n, dtype=np.uint32)
    res = {}

    def torch_loop():
        res["L"] = api.trace_paths(sc, d_rays, d_keys, DEPTH, seed)

    def wavefront():
        res["means"] = sc.trace_pixel_samples_group(d_rays, offsets, pix, DEPTH, seed=seed)

    ms = timed({"trace_paths": torch_loop, "group": wavefront}, warmup, reps)
    same = np.array_equal(api.group_means(res["L"], offsets), res["means"].cpu().numpy())
    assert same, f"{what}: trace_paths differs from the group entry"
    return {"set": what, "paths": n, "depth": DEPTH, "trace_paths_ms": ms["trace_paths"], "group_ms": ms["group"],
            "trace_paths_mpaths_s": n / ms["trace_paths"] / 1e3, "group_mpaths_s": n / ms["group"] / 1e3,
            "slowdown": ms["trace_paths"] / ms["group"], "bit_identical": same}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if rt.device_count() == 0:
        raise SystemExit("bench_scatter needs a CUDA device")
    res = {"bench": "scatter", **gpu_info(0), "warmup": args.warmup, "reps": args.reps, "rays": [], "paths": []}
    for name in ("cornell_box.json", "dupin.json", "4b"):
        sc, cam = load(name)
        tag = name.replace(".json", "")
        rays = camera_rays(cam, 2048, 2048, 1, np.random.default_rng(1))
        row, secondary = scatter_vs_nearest(f"{tag}_camera", sc, rays, args.warmup, args.reps)
        print(json.dumps(row), flush=True)
        res["rays"].append(row)
        row, _ = scatter_vs_nearest(f"{tag}_secondary", sc, secondary, args.warmup, args.reps)
        print(json.dumps(row), flush=True)
        res["rays"].append(row)
        row = paths(f"{tag}_camera_1024x1024", sc, cam, max(1, args.warmup // 2), max(3, args.reps // 2))
        print(json.dumps(row), flush=True)
        res["paths"].append(row)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
