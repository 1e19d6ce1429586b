#!/usr/bin/env python
"""Timing of rt_trace_pixel_samples_group[_device] (caller rays of many pixels in one wavefront) against the frame path.

  python tools/bench_trace_group.py [--warmup 2] [--reps 5] [--out FILE]

Prints ONE JSON line (and writes it to FILE when given).  Needs a CUDA device; reads the GPU's name and power limit
with a read-only nvidia-smi query in the same run.

1. Same paths as a frame: cornell_box 1024x1024x16 and spheres 640x480x16 (seeded random spheres), depth 8.  The
   caller rays are the pinhole camera's primary rays built on the host with vectorised numpy (uniform jitter drawn by
   numpy, so the paths are not the frame's: this is a timing, not a parity check).  Mpaths/s, host clock around work
   that ends in a device synchronise, median / min / max over the repetitions, for
     frame         rt_render_start + rt_render_wait (result left on the device)
     group_host    rt_trace_pixel_samples_group: rays uploaded from pageable host memory, means copied back; the time of
                   a pageable upload of the same rays by torch is reported beside it as the H2D share
     group_device  rt_trace_pixel_samples_group_device on rays resident in a torch tensor, torch's current stream
   plus one pass of each with rt_set_kernel_timing on (one lane; device ms per kernel class).
2. Probe-sized groups: cornell_box, 4096 groups of 10 jittered camera rays of random pixels, depth 10: one group call
   against 4096 rt_trace_pixel_samples calls.
3. A large group: 4 Mi rays as one group against the same rays as groups of 16 (device form), with the kernel
   classes' device time: the cost of k_group_resolve's serial per-group sum.
"""
from __future__ import annotations

import argparse
import json
import math
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

SEED = 2024


def gpu_info(device: int) -> dict:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(device)],
                         capture_output=True, text=True, check=True).stdout.strip()
    name, power = [s.strip() for s in out.split(",")]
    return {"gpu": name, "power_limit": power}


def camera_rays(cam, w: int, h: int, spp: int, rng, pixels=None) -> np.ndarray:
    """MultisamplerRayCaster::new / get_ray (src/camera/ray_caster.rs:30-48,100-118) for `pixels` (default: every pixel,
    in order x + y*w) x spp, sample-minor; jitter from numpy"""
    pos, dirn = np.array(cam.position.tuple()), np.array(cam.direction.tuple())
    right, up = np.array(cam.right.tuple()), np.array(cam.up.tuple())
    center = pos + dirn * cam.focal_length
    vw = math.tan(cam.fov_rad / 2.0) * cam.focal_length * 2.0
    vh = vw / (w / h)
    left_top = center - (vw / 2.0) * right + (vh / 2.0) * up
    res = vw / w
    pixel = np.repeat(np.arange(w * h, dtype=np.int64) if pixels is None else np.asarray(pixels, np.int64), spp)
    x = (pixel % w) + rng.random(pixel.shape[0])
    y = (pixel // w) + rng.random(pixel.shape[0])
    rays = np.empty((pixel.shape[0], 6))
    rays[:, :3] = pos
    for k in range(3):   # per component: keeps the temporaries at one column
        rays[:, 3 + k] = left_top[k] + (res * x) * right[k] - (res * y) * up[k] - pos[k]
    rays[:, 3:] /= np.sqrt((rays[:, 3:] ** 2).sum(axis=1))[:, None]
    return rays


def timed(fn, sync, warmup: int, reps: int) -> list:
    for _ in range(warmup):
        fn()
    sync()
    ts = []
    for _ in range(reps):
        sync()
        t0 = time.perf_counter()
        fn()
        sync()
        ts.append(time.perf_counter() - t0)
    return ts


def rate(paths: int, ts: list) -> dict:
    ms = sorted(t * 1e3 for t in ts)
    return {"mpaths_s_median": round(paths / np.median(ms) / 1e3, 1), "mpaths_s_min": round(paths / ms[-1] / 1e3, 1),
            "mpaths_s_max": round(paths / ms[0] / 1e3, 1), "ms": [round(m, 3) for m in ms]}


def kernel_ms(sc) -> dict:
    st = sc.stats()
    return {k: round(getattr(st, "ms_" + k), 3) for k in ("raygen", "extend", "march", "shade", "resolve")}


def same_paths(torch, name: str, w: int, h: int, spp: int, depth: int, warmup: int, reps: int) -> dict:
    sync = torch.cuda.synchronize
    sc = rt.Scene.from_file(os.path.join(ROOT, "scenes", name), random_spheres_seed=1)
    cam = sc.camera()
    ds = sc.device_scene(0)
    n = w * h * spp
    rays = camera_rays(cam, w, h, spp, np.random.default_rng(1))
    offsets = np.arange(0, n + 1, spp, dtype=np.uint64)
    pix = np.arange(w * h, dtype=np.uint32)
    params = api.render_params(w, h, spp, depth, SEED)

    def frame():
        api.render_start(ds, cam, params)
        api.render_wait(ds, None)

    host = lambda: sc.trace_pixel_samples_group(rays, offsets, pix, depth, seed=SEED)
    d_rays = torch.from_numpy(rays).cuda()
    device = lambda: sc.trace_pixel_samples_group(d_rays, offsets, pix, depth, seed=SEED)
    upload = lambda: torch.from_numpy(rays).to("cuda")
    out = {"scene": name, "w": w, "h": h, "spp": spp, "depth": depth, "paths": n}
    # alternate the three forms rep by rep, so that a drift of the clocks or of other work on the host hits all of them
    t = {"frame": [], "group_host": [], "group_device": [], "h2d": []}
    fns = {"frame": frame, "group_host": host, "group_device": device, "h2d": upload}
    for k, fn in fns.items():
        timed(fn, sync, warmup, 0)
    for _ in range(reps):
        for k, fn in fns.items():
            t[k] += timed(fn, sync, 0, 1)
    for k in ("frame", "group_host", "group_device"):
        out[k] = rate(n, t[k])
    h2d = float(np.median(t["h2d"])) * 1e3
    out["group_host"]["h2d_ms_median"] = round(h2d, 3)
    out["group_host"]["h2d_share"] = round(h2d / float(np.median(t["group_host"]) * 1e3), 3)
    out["device_over_frame"] = round(out["group_device"]["mpaths_s_median"] / out["frame"]["mpaths_s_median"], 3)
    # device time per kernel class, one pass each (kernel timing runs the batches on one lane)
    out["kernel_ms"] = {}
    sc.set_kernel_timing(True)
    for k, fn in (("frame", frame), ("group_device", device)):
        sc.reset_stats()
        fn()
        sync()
        out["kernel_ms"][k] = kernel_ms(sc)
    sc.set_kernel_timing(False)
    return out


def probe(torch, warmup: int, reps: int) -> dict:
    sync = torch.cuda.synchronize
    w = h = 1024
    groups, per, depth = 4096, 10, 10
    sc = rt.Scene.from_file(os.path.join(ROOT, "scenes", "cornell_box.json"), random_spheres_seed=1)
    cam = sc.camera()
    rng = np.random.default_rng(2)
    pix = rng.choice(w * h, groups, replace=False).astype(np.uint32)
    rays = camera_rays(cam, w, h, per, rng, pixels=pix)
    offsets = np.arange(0, groups * per + 1, per, dtype=np.uint64)
    group = lambda: sc.trace_pixel_samples_group(rays, offsets, pix, depth, seed=SEED)

    def one_by_one():
        for g in range(groups):
            sc.trace_pixel_samples(rays[g * per:(g + 1) * per], depth, seed=SEED, pixel_index=int(pix[g]))

    tg = timed(group, sync, warmup, reps)
    tl = timed(one_by_one, sync, 1, max(2, reps // 2))
    mg, ml = float(np.median(tg)) * 1e3, float(np.median(tl)) * 1e3
    return {"scene": "cornell_box.json", "groups": groups, "rays_per_group": per, "depth": depth,
            "group_call_ms": [round(x * 1e3, 3) for x in sorted(tg)],
            "per_pixel_calls_ms": [round(x * 1e3, 1) for x in sorted(tl)],
            "speedup_median": round(ml / mg, 1)}


def large_group(torch, warmup: int, reps: int) -> dict:
    """one group of 4 Mi rays against the same rays as 256 Ki groups of 16 (device form, cornell_box, depth 8):
    k_group_resolve sums a group's slice of a batch in ONE thread, serially, so a group much larger than a pixel's
    sample count makes the resolve a long serial loop"""
    sync = torch.cuda.synchronize
    n, per, depth = 1 << 22, 16, 8
    sc = rt.Scene.from_file(os.path.join(ROOT, "scenes", "cornell_box.json"), random_spheres_seed=1)
    cam = sc.camera()
    rng = np.random.default_rng(3)
    pix = rng.choice(1024 * 1024, n // per, replace=False)
    d_rays = torch.from_numpy(camera_rays(cam, 1024, 1024, per, rng, pixels=pix)).cuda()
    out = {"scene": "cornell_box.json", "rays": n, "depth": depth}
    for name, offsets, pi in (("one_group", np.array([0, n], np.uint64), np.array([7], np.uint32)),
                              ("groups_of_16", np.arange(0, n + 1, per, dtype=np.uint64), pix.astype(np.uint32))):
        fn = lambda: sc.trace_pixel_samples_group(d_rays, offsets, pi, depth, seed=SEED)
        out[name] = rate(n, timed(fn, sync, warmup, reps))
        sc.set_kernel_timing(True)
        sc.reset_stats()
        fn()
        sync()
        out[name]["kernel_ms"] = kernel_ms(sc)
        sc.set_kernel_timing(False)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if rt.device_count() == 0 or not torch.cuda.is_available():
        raise SystemExit("bench_trace_group needs a CUDA device")
    torch.cuda.set_device(0)
    result = {"tool": "bench_trace_group", **gpu_info(0),
              "same_paths": [same_paths(torch, "cornell_box.json", 1024, 1024, 16, 8, args.warmup, args.reps),
                             same_paths(torch, "spheres.json", 640, 480, 16, 8, args.warmup, args.reps)],
              "probe": probe(torch, args.warmup, args.reps),
              "large_group": large_group(torch, args.warmup, args.reps)}
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
