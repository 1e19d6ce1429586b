#!/usr/bin/env python
"""Views frames (rt_render_start_views) against one frame per camera.

  python tools/bench_views.py [--warmup 1] [--reps 3] [--out FILE]

Prints ONE JSON line (and writes it to FILE when given).  Needs a CUDA device; reads the GPU's name and power limit
with a read-only nvidia-smi query in the same run.  Times are a host clock around the whole job (start + wait, the
frames left on the device), median over the repetitions, the ways alternated rep by rep.

1. Small frames, where the fixed cost of a frame (five launches per bounce level, the drain of the thin deep levels, the
   host's turn-around) is a large share: spheres 640x480 at depth 8 with 1 and 4 spp, and the bins' setting,
   cornell_box 1600x900 at 1 spp and depth 50.  Each at V = 1, 2, 8 and 32 orbit views (tools/render.py --orbit),
   rendered three ways: one views frame; V rt_render_start frames on one handle; DistributedRenderer.render_jobs on
   one rank (two frames in flight on two handles; it also copies every frame to pinned host memory).  Reported: ms
   per view and Mpaths/s of each way, and whether the views frame equals the V frames bit for bit.
2. The cost of the unfused level 0 (k_raygen_views + k_extend instead of the raygen k_extend): V = 1 at bench.py
   config 3's size (cornell_box 1024x1024, 256 spp, depth 8) against rt_render_start, and one frame of each with
   kernel timing on.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

import rs_pathtracing_b200 as rt  # noqa: E402
from rs_pathtracing_b200 import api  # noqa: E402
from bench_adaptive import alternate, gpu_info  # noqa: E402

SEED = 2024
SMALL = [("spheres.json", 640, 480, 1, 8), ("spheres.json", 640, 480, 4, 8), ("cornell_box.json", 1600, 900, 1, 50)]
VIEWS = [1, 2, 8, 32]


def load(name):
    sc = rt.Scene.from_file(os.path.join(ROOT, "scenes", name), random_spheres_seed=1)
    return sc, sc.camera()


def views_frame(hd, cams, w, h, spp, depth, buf=None):
    api.render_start_views(hd, cams, api.render_params(w, h, spp, depth, SEED))
    api.render_wait(hd, buf)


def frames(hd, cams, w, h, spp, depth, buf=None):
    for v, c in enumerate(cams):
        api.render_start(hd, c, api.render_params(w, h, spp, depth, SEED))
        api.render_wait(hd, None if buf is None else buf[v])


def breakdown(sc, fn) -> dict:
    sc.set_kernel_timing(True, 0)
    sc.reset_stats(0)
    fn()
    s = sc.stats(0)
    sc.set_kernel_timing(False, 0)
    return {"frame_ms": round(s.last_frame_ms, 3), "raygen": round(s.ms_raygen, 3), "extend": round(s.ms_extend, 3),
            "march": round(s.ms_march, 3), "shade": round(s.ms_shade, 3), "resolve": round(s.ms_resolve, 3)}


def small_frames(warmup: int, reps: int) -> list:
    from rs_pathtracing_b200.distributed import DistributedRenderer
    out = []
    for name, w, h, spp, depth in SMALL:
        sc, cam = load(name)
        hd = sc.device_scene(0)
        dr = DistributedRenderer(sc, depth, seed=SEED, device=0)
        for V in VIEWS:
            cams = api.orbit_cameras(cam, V)
            a, b = np.zeros((V, h, w, 3)), np.zeros((V, h, w, 3))
            views_frame(hd, cams, w, h, spp, depth, a)
            frames(hd, cams, w, h, spp, depth, b)
            jobs = [(c, w, h, spp) for c in cams]
            t = alternate({"views": lambda: views_frame(hd, cams, w, h, spp, depth),
                           "frames": lambda: frames(hd, cams, w, h, spp, depth),
                           "render_jobs": lambda: dr.render_jobs(jobs)}, warmup, reps)
            paths = V * w * h * spp
            row = {"scene": name, "w": w, "h": h, "spp": spp, "depth": depth, "n_views": V,
                   "identical": bool(np.array_equal(a, b))}
            for k, ms in t.items():
                row[k] = {"ms_per_view": round(ms / V, 3), "mpaths_s": round(paths / ms / 1e3, 1)}
            row["views_speedup_vs_frames"] = round(t["frames"] / t["views"], 3)
            row["views_speedup_vs_render_jobs"] = round(t["render_jobs"] / t["views"], 3)
            out.append(row)
            print(json.dumps(row), file=sys.stderr, flush=True)
    return out


def level0_cost(warmup: int, reps: int) -> dict:
    w, h, spp, depth = 1024, 1024, 256, 8
    sc, cam = load("cornell_box.json")
    hd = sc.device_scene(0)
    a, b = np.zeros((1, h, w, 3)), np.zeros((1, h, w, 3))
    views_frame(hd, [cam], w, h, spp, depth, a)
    frames(hd, [cam], w, h, spp, depth, b)
    t = alternate({"views": lambda: views_frame(hd, [cam], w, h, spp, depth),
                   "frame": lambda: frames(hd, [cam], w, h, spp, depth)}, warmup, reps)
    paths = w * h * spp
    return {"scene": "cornell_box.json", "w": w, "h": h, "spp": spp, "depth": depth,
            "identical": bool(np.array_equal(a, b)),
            "views_ms": round(t["views"], 2), "frame_ms": round(t["frame"], 2),
            "views_mpaths_s": round(paths / t["views"] / 1e3, 1), "frame_mpaths_s": round(paths / t["frame"] / 1e3, 1),
            "views_over_frame": round(t["views"] / t["frame"], 4),
            "views_kernels": breakdown(sc, lambda: views_frame(hd, [cam], w, h, spp, depth)),
            "frame_kernels": breakdown(sc, lambda: frames(hd, [cam], w, h, spp, depth))}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if rt.device_count() == 0:
        raise SystemExit("bench_views needs a CUDA device")
    res = {"tool": "bench_views", **gpu_info(0), "seed": SEED, "warmup": a.warmup, "reps": a.reps,
           "small_frames": small_frames(a.warmup, a.reps), "level0_cfg3": level0_cost(a.warmup, a.reps)}
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
