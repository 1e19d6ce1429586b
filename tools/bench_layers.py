#!/usr/bin/env python
"""Layers frames (rt_render_start_layers) against the plain frame of the same camera and parameters.

  python tools/bench_layers.py [--warmup 1] [--reps 3] [--out FILE]

Prints ONE JSON line (and writes it to FILE when given).  Needs a CUDA device; reads the GPU's name and power limit
with a read-only nvidia-smi query in the same run.  Times are a host clock around the whole frame (start + wait, the
frame and the layers left on the device), median over the repetitions, the ways alternated rep by rep.  Each case also
runs one frame of each way with kernel timing on, for the resolve's own cost (k_resolve against k_resolve_layers and
the layers' k_assemble_layers).

Cases: bench.py config 3's frame at the reference bins' depth (cornell_box 1024x1024, 256 spp, depth 50), config 4b
(detached_materials with every material kind, 1920x1080, 256 spp, depth 8) and dupin (960x540, 64 spp, depth 50: a
ray-marched surface), each at n_layers 1, 4 and max_depth + 1.  Reported: ms, Mpaths/s, the overhead over the plain
frame, whether the frame equals the plain frame bit for bit, and each layer's share of the mean luminance.
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
CASES = [("3", "cornell_box.json", 1024, 1024, 256, 50), ("4b", "detached_materials.json", 1920, 1080, 256, 8),
         ("dupin", "dupin.json", 960, 540, 64, 50)]


def load(cfg, name):
    if cfg in ("3", "4b"):
        return load_config_scene(cfg)
    sc = rt.Scene.from_file(os.path.join(ROOT, "scenes", name), random_spheres_seed=1)
    return sc, sc.camera()


def plain(hd, cam, w, h, spp, depth, buf=None):
    api.render_start(hd, cam, api.render_params(w, h, spp, depth, SEED))
    api.render_wait(hd, buf)


def layers(hd, cam, w, h, spp, depth, n, buf=None):
    api.render_start_layers(hd, cam, api.render_params(w, h, spp, depth, SEED), n)
    api.render_wait(hd, buf)


def resolve_ms(sc, fn) -> dict:
    sc.set_kernel_timing(True, 0)
    sc.reset_stats(0)
    fn()
    s = sc.stats(0)
    sc.set_kernel_timing(False, 0)
    return {"frame_ms": round(s.last_frame_ms, 3), "resolve_ms": round(s.ms_resolve, 3)}


def luminance_share(frame, ls):
    y = lambda a: (0.2126 * a[..., 0] + 0.7152 * a[..., 1]) + 0.0722 * a[..., 2]
    total = float(np.mean(y(frame)))
    return [round(float(np.mean(y(l))) / total, 6) if total else 0.0 for l in ls]


def case(cfg, name, w, h, spp, depth, warmup, reps) -> dict:
    sc, cam = load(cfg, name)
    hd = sc.device_scene(0)
    counts = sorted({1, 4, depth + 1})
    ref = np.zeros((h, w, 3))
    plain(hd, cam, w, h, spp, depth, ref)
    row = {"case": cfg, "scene": name, "w": w, "h": h, "spp": spp, "depth": depth, "layers": {}}
    fns = {"plain": lambda: plain(hd, cam, w, h, spp, depth)}
    for n in counts:
        fns[n] = (lambda n=n: layers(hd, cam, w, h, spp, depth, n))
    t = alternate(fns, warmup, reps)
    paths = w * h * spp
    row["plain"] = {"ms": round(t["plain"], 2), "mpaths_s": round(paths / t["plain"] / 1e3, 1),
                    **resolve_ms(sc, fns["plain"])}
    for n in counts:
        frame = np.zeros((h, w, 3))
        layers(hd, cam, w, h, spp, depth, n, frame)
        ls = api.render_layers(hd)
        row["layers"][str(n)] = {"ms": round(t[n], 2), "mpaths_s": round(paths / t[n] / 1e3, 1),
                                 "overhead": round(t[n] / t["plain"] - 1.0, 4),
                                 "frame_identical": bool(np.array_equal(frame, ref)),
                                 "luminance_share": luminance_share(frame, ls), **resolve_ms(sc, fns[n])}
        del ls
    print(json.dumps(row), file=sys.stderr, flush=True)
    return row


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if rt.device_count() == 0:
        raise SystemExit("bench_layers needs a CUDA device")
    res = {"tool": "bench_layers", **gpu_info(0), "seed": SEED, "warmup": a.warmup, "reps": a.reps,
           "cases": [case(*c, a.warmup, a.reps) for c in CASES]}
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
