#!/usr/bin/env python
"""Counts frames (rt_render_start_counts) against uniform and adaptive frames.

  python tools/bench_counts.py [--warmup 1] [--reps 3] [--out FILE]

Prints ONE JSON line (and writes it to FILE when given).  Needs a CUDA device; reads the GPU's name and power limit
with a read-only nvidia-smi query in the same run.  Times are a host clock around start + wait (the frame left on the
device), median over the repetitions, the variants alternated rep by rep.

1. uniform maps against rt_render_start: bench.py config 3 (cornell_box 1024x1024, 256 spp, depth 8) and spheres
   640x480x256: Mpaths/s of both, whether the frames are identical, and one frame of each with kernel timing on
   (the loader counts as raygen, k_counts_resolve as resolve) plus the start call's host time.
2. adaptive replay, with tools/bench_adaptive.py's settings (min 8, at most 256; rel 0.05 and 0.02 on cornell_box
   1024x1024, 0.01 on spheres 640x480): the adaptive frame, the counts frame of its counts (which must be the same
   frame) and the uniform frame of (about) equal paths.
3. the replayed cornell_box map (rel 0.05) on a multi-device handle over every GPU against one GPU, and each shard's
   device time rendered alone (slowest against the mean); "not measured" with one GPU.
4. the host time of the start call for a random map (counts 0..16) at 3840x2160: the first call on a fresh handle and
   the median of the following ones, against rt_render_start's.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

import rs_pathtracing_b200 as rt  # noqa: E402
from rs_pathtracing_b200 import api  # noqa: E402
from bench_adaptive import alternate, gpu_info  # noqa: E402

SEED, DEPTH, MIN, SPP = 2024, 8, 8, 256


def load(name):
    sc = rt.Scene.from_file(os.path.join(ROOT, "scenes", name), random_spheres_seed=1)
    return sc, sc.camera()


def uniform(hd, cam, w, h, spp, buf=None):
    api.render_start(hd, cam, api.render_params(w, h, spp, DEPTH, SEED))
    api.render_wait(hd, buf)


def counts_frame(hd, cam, counts, cap, buf=None):
    h, w = counts.shape
    api.render_start_counts(hd, cam, api.render_params(w, h, cap, DEPTH, SEED), counts)
    api.render_wait(hd, buf)


def adaptive(hd, cam, w, h, rel, buf=None):
    api.render_start_adaptive(hd, cam, api.render_params(w, h, SPP, DEPTH, SEED), MIN, rel)
    api.render_wait(hd, buf)


def breakdown(sc, fn) -> dict:
    sc.set_kernel_timing(True, 0)
    sc.reset_stats(0)
    fn()
    s = sc.stats(0)
    sc.set_kernel_timing(False, 0)
    return {"frame_ms": round(s.last_frame_ms, 3), "raygen": round(s.ms_raygen, 3), "extend": round(s.ms_extend, 3),
            "march": round(s.ms_march, 3), "shade": round(s.ms_shade, 3), "resolve": round(s.ms_resolve, 3)}


def start_call_ms(fn, reps=5):
    t = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        t.append((time.perf_counter() - t0) * 1e3)
    return t


def uniform_maps(warmup, reps):
    out = []
    for name, w, h in (("cornell_box.json", 1024, 1024), ("spheres.json", 640, 480)):
        sc, cam = load(name)
        hd = sc.device_scene(0)
        full = np.full((h, w), SPP, np.uint32)
        a, b = np.zeros((h, w, 3)), np.zeros((h, w, 3))
        uniform(hd, cam, w, h, SPP, a)
        counts_frame(hd, cam, full, SPP, b)
        t = alternate({"render_start": lambda: uniform(hd, cam, w, h, SPP),
                       "counts": lambda: counts_frame(hd, cam, full, SPP)}, warmup, reps)
        paths = w * h * SPP

        def start_only(fn):
            t0 = time.perf_counter()
            fn()
            dt = (time.perf_counter() - t0) * 1e3
            api.render_wait(hd, None)
            return dt

        s_u = start_only(lambda: api.render_start(hd, cam, api.render_params(w, h, SPP, DEPTH, SEED)))
        s_c = start_only(lambda: api.render_start_counts(hd, cam, api.render_params(w, h, SPP, DEPTH, SEED), full))
        out.append({"scene": name, "w": w, "h": h, "spp": SPP, "depth": DEPTH, "identical": bool(np.array_equal(a, b)),
                    "render_start": {"ms": round(t["render_start"], 3),
                                     "mpaths_s": round(paths / t["render_start"] / 1e3, 1)},
                    "counts": {"ms": round(t["counts"], 3), "mpaths_s": round(paths / t["counts"] / 1e3, 1)},
                    "ratio": round(t["render_start"] / t["counts"], 4),
                    "start_call_ms": {"render_start": round(s_u, 3), "counts": round(s_c, 3)},
                    "kernel_ms_render_start": breakdown(sc, lambda: uniform(hd, cam, w, h, SPP)),
                    "kernel_ms_counts": breakdown(sc, lambda: counts_frame(hd, cam, full, SPP))})
    return out


def replay(warmup, reps):
    out, maps = [], {}
    for name, w, h, rel in (("cornell_box.json", 1024, 1024, 0.05), ("cornell_box.json", 1024, 1024, 0.02),
                            ("spheres.json", 640, 480, 0.01)):
        sc, cam = load(name)
        hd = sc.device_scene(0)
        fa, fc = np.zeros((h, w, 3)), np.zeros((h, w, 3))
        adaptive(hd, cam, w, h, rel, fa)
        counts, _ = api.render_pixel_stats(hd)
        counts_frame(hd, cam, counts, SPP, fc)
        paths = int(counts.sum(dtype=np.uint64))
        u_spp = max(1, int(round(paths / (w * h))))
        t = alternate({"adaptive": lambda: adaptive(hd, cam, w, h, rel),
                       "counts_replay": lambda: counts_frame(hd, cam, counts, SPP),
                       "uniform_equal_paths": lambda: uniform(hd, cam, w, h, u_spp)}, warmup, reps)
        u_paths = w * h * u_spp
        maps[(name, rel)] = counts
        out.append({"scene": name, "w": w, "h": h, "rel_error": rel, "min_samples": MIN, "samples_number": SPP,
                    "paths": paths, "replay_identical": bool(np.array_equal(fa, fc)),
                    "adaptive": {"ms": round(t["adaptive"], 3), "mpaths_s": round(paths / t["adaptive"] / 1e3, 1)},
                    "counts_replay": {"ms": round(t["counts_replay"], 3),
                                      "mpaths_s": round(paths / t["counts_replay"] / 1e3, 1)},
                    "uniform_equal_paths": {"spp": u_spp, "paths": u_paths, "ms": round(t["uniform_equal_paths"], 3),
                                            "mpaths_s": round(u_paths / t["uniform_equal_paths"] / 1e3, 1)},
                    "replay_saves_vs_adaptive": round(1.0 - t["counts_replay"] / t["adaptive"], 4),
                    "replay_vs_uniform_time_per_path": round((t["counts_replay"] / paths) / (t["uniform_equal_paths"] / u_paths), 4)})
    return out, maps[("cornell_box.json", 0.05)]


def multi(counts, warmup, reps):
    n = rt.device_count()
    if n < 2:
        return {"measured": False, "reason": f"not measured: {n} GPU visible"}
    h, w = counts.shape
    sc, cam = load("cornell_box.json")
    one, hm = sc.device_scene(0), sc.device_scene_multi(list(range(n)))
    a, b = np.zeros((h, w, 3)), np.zeros((h, w, 3))
    counts_frame(one, cam, counts, SPP, a)
    counts_frame(hm, cam, counts, SPP, b)
    t = alternate({"one_gpu": lambda: counts_frame(one, cam, counts, SPP),
                   "all_gpus": lambda: counts_frame(hm, cam, counts, SPP)}, warmup, reps)
    shard_ms = []
    for k in range(n):   # each shard alone on its own device (device time of the shard's frame)
        hk = sc.device_scene(k)
        p = api.render_params(w, h, SPP, DEPTH, SEED, n, k, tile=32)
        for _ in range(2):
            api.render_start_counts(hk, cam, p, counts)
            api.render_wait(hk, None)
        shard_ms.append(sc.stats(k).last_frame_ms)
    return {"measured": True, "gpus": n, "identical": bool(np.array_equal(a, b, equal_nan=True)),
            "one_gpu_ms": round(t["one_gpu"], 3), "all_gpus_ms": round(t["all_gpus"], 3),
            "speedup": round(t["one_gpu"] / t["all_gpus"], 3), "shard_ms": [round(x, 3) for x in shard_ms],
            "slowest_over_mean": round(max(shard_ms) / (sum(shard_ms) / n), 4)}


def start_time_4k():
    w, h, cap = 3840, 2160, 16
    counts = np.random.default_rng(1).integers(0, cap + 1, (h, w)).astype(np.uint32)
    sc, cam = load("cornell_box.json")
    hd = sc.device_scene(0)
    p = api.render_params(w, h, cap, DEPTH, SEED)
    times = []
    for _ in range(6):
        t0 = time.perf_counter()
        api.render_start_counts(hd, cam, p, counts)
        times.append((time.perf_counter() - t0) * 1e3)
        api.render_wait(hd, None)
    u = []
    for _ in range(5):
        t0 = time.perf_counter()
        api.render_start(hd, cam, p)
        u.append((time.perf_counter() - t0) * 1e3)
        api.render_wait(hd, None)
    return {"w": w, "h": h, "counts": f"uniform random 0..{cap}", "first_call_ms": round(times[0], 3),
            "median_ms": round(float(np.median(times[1:])), 3), "render_start_median_ms": round(float(np.median(u[1:])), 3),
            "method": "host computes the owned pixels' u64 path offsets and uploads them (8 B per pixel, pageable)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if rt.device_count() == 0:
        raise SystemExit("no CUDA device: counts frames run on the GPU only")
    res = {"bench": "counts", **gpu_info(0), "uniform_maps": uniform_maps(a.warmup, a.reps)}
    res["adaptive_replay"], cornell_map = replay(a.warmup, a.reps)
    res["multi_device"] = multi(cornell_map, a.warmup, a.reps)
    res["start_call_4k"] = start_time_4k()
    line = json.dumps(res)
    print(line, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
