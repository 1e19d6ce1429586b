#!/usr/bin/env python
"""Features frames (rt_render_start_features) against the plain frame of the same camera and parameters.

  python tools/bench_features.py [--warmup 1] [--reps 3] [--out FILE]

Prints ONE JSON line (and writes it to FILE when given).  Needs a CUDA device; reads the GPU's name and power limit
with a read-only nvidia-smi query in the same run.  Times are a host clock around the whole frame (start + wait, the
frame and the features left on the device), median over the repetitions, the ways alternated rep by rep.  Each case
also runs one frame of each way with kernel timing on, for the cost of the feature kernels (k_features_path counts as
shade, k_features_resolve and k_assemble_features as resolve).

Cases: bench.py config 3's frame (cornell_box 1024x1024, 256 spp, depth 8), config 4b (detached_materials with every
material kind, 1920x1080, 256 spp, depth 8) and dupin (960x540, 64 spp, depth 50: a ray-marched surface).  Reported:
ms, Mpaths/s, the overhead over the plain frame, whether the frame equals the plain frame bit for bit, and the mean
coverage.
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
from bench import load_config_scene  # noqa: E402

SEED = 2024
CASES = [("3", "cornell_box.json", 1024, 1024, 256, 8), ("4b", "detached_materials.json", 1920, 1080, 256, 8),
         ("dupin", "dupin.json", 960, 540, 64, 50)]


def load(cfg, name):
    if cfg in ("3", "4b"):
        return load_config_scene(cfg)
    sc = rt.Scene.from_file(os.path.join(ROOT, "scenes", name), random_spheres_seed=1)
    return sc, sc.camera()


def plain(hd, cam, w, h, spp, depth, buf=None):
    api.render_start(hd, cam, api.render_params(w, h, spp, depth, SEED))
    api.render_wait(hd, buf)


def features(hd, cam, w, h, spp, depth, buf=None):
    api.render_start_features(hd, cam, api.render_params(w, h, spp, depth, SEED))
    api.render_wait(hd, buf)


def kernel_ms(sc, fn) -> dict:
    sc.set_kernel_timing(True, 0)
    sc.reset_stats(0)
    fn()
    s = sc.stats(0)
    sc.set_kernel_timing(False, 0)
    return {"frame_ms": round(s.last_frame_ms, 3), "shade_ms": round(s.ms_shade, 3), "resolve_ms": round(s.ms_resolve, 3)}


def case(cfg, name, w, h, spp, depth, warmup, reps) -> dict:
    sc, cam = load(cfg, name)
    hd = sc.device_scene(0)
    ref = np.zeros((h, w, 3))
    plain(hd, cam, w, h, spp, depth, ref)
    fns = {"plain": lambda: plain(hd, cam, w, h, spp, depth), "features": lambda: features(hd, cam, w, h, spp, depth)}
    t = alternate(fns, warmup, reps)
    paths = w * h * spp
    frame = np.zeros((h, w, 3))
    features(hd, cam, w, h, spp, depth, frame)
    feats = api.render_features(hd)
    row = {"case": cfg, "scene": name, "w": w, "h": h, "spp": spp, "depth": depth,
           "plain": {"ms": round(t["plain"], 2), "mpaths_s": round(paths / t["plain"] / 1e3, 1),
                     **kernel_ms(sc, fns["plain"])},
           "features": {"ms": round(t["features"], 2), "mpaths_s": round(paths / t["features"] / 1e3, 1),
                        "overhead": round(t["features"] / t["plain"] - 1.0, 4),
                        "frame_identical": bool(np.array_equal(frame, ref)),
                        "mean_coverage": round(float(feats["coverage"].mean()), 6), **kernel_ms(sc, fns["features"])}}
    print(json.dumps(row), file=sys.stderr, flush=True)
    return row


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if rt.device_count() == 0:
        raise SystemExit("bench_features needs a CUDA device")
    res = {"tool": "bench_features", **gpu_info(0), "seed": SEED, "warmup": a.warmup, "reps": a.reps,
           "cases": [case(*c, a.warmup, a.reps) for c in CASES]}
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
