#!/usr/bin/env python
"""Adaptive sampling (rt_render_start_adaptive) against uniform frames: cost, paths and error.

  python tools/bench_adaptive.py [--warmup 1] [--reps 3] [--out FILE]

Prints ONE JSON line (and writes it to FILE when given).  Needs a CUDA device; reads the GPU's name and power limit
with a read-only nvidia-smi query in the same run.  Times are a host clock around start + wait (the frame left on the
device), median over the repetitions, the variants alternated rep by rep.

1. cornell_box 1024x1024 and spheres 640x480 (seeded random spheres), depth 8, min_samples 8, at most 256 samples,
   rel_error in {0.05, 0.02, 0.01}: paths traced, ms, Mpaths/s, and the RMSE against a 4096-spp reference frame of
   another seed, in display space (sqrt, clamped to [0, 0.999] as the bins' tone map) and in linear space (clamped
   to [0, 4]); the same for the uniform frame with (about) the same total paths, and for the uniform 256-spp frame.
   boundary_share = 1 - (paths / uniform rate) / adaptive time: the share of the adaptive frame spent beyond what its
   paths cost in a uniform frame (drained wavefront tails at pass boundaries, selects, empty launches).
2. bench.py config 3 (cornell_box 1024x1024x256): min_samples == samples_number against rt_render_start (the same
   frame plus the moments), and min 8 / at most 256 with a rel_error so large that every pixel stops after pass 0
   against the uniform 8-spp frame: the five refinement passes are planned, selected and launched, and find nothing
   to do (the empty launches).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import rs_pathtracing_b200 as rt  # noqa: E402
from rs_pathtracing_b200 import api  # noqa: E402

SEED, REF_SEED, DEPTH = 2024, 99, 8


def gpu_info(device: int) -> dict:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(device)],
                         capture_output=True, text=True, check=True).stdout.strip()
    name, power = [s.strip() for s in out.split(",")]
    return {"gpu": name, "power_limit": power}


def display(f):
    return np.clip(np.sqrt(np.maximum(f, 0.0)), 0.0, 0.999)


def rmse(a, b):
    return {"display": float(np.sqrt(np.mean((display(a) - display(b)) ** 2))),
            "linear": float(np.sqrt(np.mean((np.clip(a, 0, 4) - np.clip(b, 0, 4)) ** 2)))}


class Frames:
    def __init__(self, sc, cam, w, h):
        self.ds, self.cam, self.w, self.h = sc.device_scene(0), cam, w, h

    def uniform(self, spp, seed=SEED, buf=None):
        api.render_start(self.ds, self.cam, api.render_params(self.w, self.h, spp, DEPTH, seed))
        api.render_wait(self.ds, buf)

    def adaptive(self, spp, mn, rel, buf=None):
        api.render_start_adaptive(self.ds, self.cam, api.render_params(self.w, self.h, spp, DEPTH, SEED), mn, rel)
        api.render_wait(self.ds, buf)


def alternate(fns: dict, warmup: int, reps: int) -> dict:
    for fn in fns.values():
        for _ in range(warmup):
            fn()
    t = {k: [] for k in fns}
    for _ in range(reps):
        for k, fn in fns.items():
            t0 = time.perf_counter()
            fn()
            t[k].append((time.perf_counter() - t0) * 1e3)
    return {k: float(np.median(v)) for k, v in t.items()}


def quality(name: str, w: int, h: int, warmup: int, reps: int, mn=8, spp=256) -> dict:
    sc = rt.Scene.from_file(os.path.join(ROOT, "scenes", name), random_spheres_seed=1)
    cam = sc.camera()
    F = Frames(sc, cam, w, h)
    ref = np.zeros((h, w, 3))
    F.uniform(4096, seed=REF_SEED, buf=ref)
    out = {"scene": name, "w": w, "h": h, "depth": DEPTH, "min_samples": mn, "samples_number": spp,
           "reference_spp": 4096, "cases": []}
    full = np.zeros((h, w, 3))
    t_full = alternate({"u": lambda: F.uniform(spp, buf=None)}, warmup, reps)["u"]
    F.uniform(spp, buf=full)
    out["uniform_max"] = {"spp": spp, "paths": w * h * spp, "ms": round(t_full, 3),
                          "mpaths_s": round(w * h * spp / t_full / 1e3, 1), "rmse": rmse(full, ref)}
    for rel in (0.05, 0.02, 0.01):
        frame = np.zeros((h, w, 3))
        F.adaptive(spp, mn, rel, buf=frame)
        counts, _ = api.render_pixel_stats(F.ds)
        paths = int(counts.sum())
        u_spp = max(1, int(round(paths / (w * h))))
        uni = np.zeros((h, w, 3))
        F.uniform(u_spp, buf=uni)
        t = alternate({"adaptive": lambda: F.adaptive(spp, mn, rel), "uniform": lambda: F.uniform(u_spp)}, warmup, reps)
        u_paths = w * h * u_spp
        u_rate = u_paths / t["uniform"]
        hist = {int(k): int(v) for k, v in zip(*np.unique(counts, return_counts=True))}
        out["cases"].append({
            "rel_error": rel,
            "adaptive": {"paths": paths, "mean_spp": round(paths / (w * h), 2), "ms": round(t["adaptive"], 3),
                         "mpaths_s": round(paths / t["adaptive"] / 1e3, 1), "rmse": rmse(frame, ref),
                         "counts": hist},
            "uniform_equal_paths": {"spp": u_spp, "paths": u_paths, "ms": round(t["uniform"], 3),
                                    "mpaths_s": round(u_rate / 1e3, 1), "rmse": rmse(uni, ref)},
            "boundary_share": round(1.0 - (paths / u_rate) / t["adaptive"], 3),
        })
    return out


def overhead(warmup: int, reps: int) -> dict:
    w, h, spp = 1024, 1024, 256
    sc = rt.Scene.from_file(os.path.join(ROOT, "scenes", "cornell_box.json"), random_spheres_seed=1)
    F = Frames(sc, sc.camera(), w, h)
    t = alternate({"render_start": lambda: F.uniform(spp), "adaptive_min_eq_max": lambda: F.adaptive(spp, spp, 0.0)},
                  warmup, reps)
    e = alternate({"render_start_8spp": lambda: F.uniform(8), "adaptive_all_stop_at_8": lambda: F.adaptive(spp, 8, 1e300)},
                  warmup, reps)
    counts, _ = api.render_pixel_stats(F.ds)
    assert (counts == 8).all()
    sc.reset_stats()
    F.adaptive(spp, 8, 1e300)
    launches_empty = sc.stats().kernel_launches
    sc.reset_stats()
    F.uniform(8)
    launches_8 = sc.stats().kernel_launches
    return {"config": "3", "scene": "cornell_box.json", "w": w, "h": h, "depth": DEPTH,
            "min_eq_max": {k: round(v, 3) for k, v in t.items()},
            "min_eq_max_overhead": round(t["adaptive_min_eq_max"] / t["render_start"] - 1.0, 4),
            "empty_passes": {**{k: round(v, 3) for k, v in e.items()},
                             "extra_ms": round(e["adaptive_all_stop_at_8"] - e["render_start_8spp"], 3),
                             "launches": launches_empty, "launches_uniform_8spp": launches_8}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if rt.device_count() == 0:
        raise SystemExit("bench_adaptive needs a CUDA device")
    result = {"tool": "bench_adaptive", **gpu_info(0),
              "quality": [quality("cornell_box.json", 1024, 1024, args.warmup, args.reps),
                          quality("spheres.json", 640, 480, args.warmup, args.reps)],
              "overhead": overhead(args.warmup, args.reps)}
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
