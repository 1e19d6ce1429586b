#!/usr/bin/env python
"""bench.py — Mpaths/s (pixels x spp / s) of the path-tracing hot path.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 1|2|3|4a|4b|5]
                  [--dump-outputs DIR]

A step is one frame of the chosen BASELINE.json configuration (default 3, the one the metric is quoted on:
scenes/cornell_box.json + seeded random spheres = 492 shapes, 1024 x 1024, 256 spp, max depth 8); config 2 is the
batched nearest-hit kernel on 1 Mi rays (Mrays/s).  One process per GPU (`--gpus N` without a torchrun environment
re-launches itself under torchrun); a frame is sharded by interleaved 32x32 tiles and gathered with one NCCL
exchange, so total work is fixed as N grows ("strong" scaling).

Output: ONE JSON line on rank 0 (the task contract): value = device-timed whole-job throughput with the scene
resident, e2e = the same through the Renderer API with host buffers, roofline for the kernel with the largest
share of the step (an ISSUE-bound FP64 path: lane-weighted issue utilisation from the committed ncu capture of this
build, executed FP64 / FP32 rates measured live; HBM traffic beside it), cpu_baseline = the oracle's threaded
renderer (C++ restatement of the reference, BVH like Scene::new builds) on a bounded sample.

`--impl reference` runs ONLY the oracle (liboracle.so) on the flattened scene files under oracle/scenes/ -- it
imports nothing of the product package and loads none of its libraries.

`--dump-outputs DIR` writes what the timed path returned in its last timed step as DIR/<name>.npy (float64, see
dump_outputs): the frame of configs 1, 3, 4a, 4b, 5 or the nearest-hit records of config 2.  Scenes, rays and RNG
seeds are fixed, so two builds run with the same arguments can be compared output for output.  Nothing is written
to the source tree.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True   # the benchmark runs from a tree it must leave as it found it (possibly read-only)
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SCENE_SEED, RNG_SEED, DEPTH = 1, 2024, 8
CONFIGS = {
    "1": dict(scene="spheres.json", w=640, h=480, spp=16,
              workload="scenes/spheres.json +481 seeded random spheres (488 shapes), 640x480, 16 spp, max depth 8"),
    "2": dict(scene=None, rays=1 << 20,
              workload="bench trio {unit Sphere, unit Cube, Heart step 0.01} x 1 Mi rays of the "
                       "benches/bench_intersections.rs recipe (about half miss), cull tree + exact-skip marching"),
    "3": dict(scene="cornell_box.json", w=1024, h=1024, spp=256,
              workload="scenes/cornell_box.json +481 seeded random spheres (492 shapes), 1024x1024, 256 spp, max depth 8"),
    "4a": dict(scene="detached_materials.json", w=1920, h=1080, spp=256,
               workload="scenes/detached_materials.json as shipped +481 seeded random spheres (488 shapes), 1920x1080, "
                        "256 spp, max depth 8"),
    "4b": dict(scene="detached_materials.json", w=1920, h=1080, spp=256,
               workload="scenes/detached_materials.json, every material / texture kind assigned, camera looking at the "
                        "origin (SURVEY 8d cfg 4b), 1920x1080, 256 spp, max depth 8"),
    "5": dict(scene="dupin.json", w=3840, h=2160, spp=1024,
              workload="scenes/dupin.json (re-authored in the current schema) +481 seeded random spheres (486 shapes), "
                       "3840x2160, 1024 spp, max depth 8"),
}

# Work per unit, counted on the reference's formulation (SURVEY 8d; DESIGN.md 5):
FLOPS_PER_SHAPE_TEST = 52      # ray -> object space (33) + unit-sphere discriminant (19), FP64
FLOPS_PER_CULL_TEST = 20       # executed FP32 flops of one conservative ball pre-test (rt_cull.cuh: 3 sub, 9 FMA, 1 mul, 1 add)
FLOPS_PER_MARCH_STEP = 22      # t/p advance (7) + Heart polynomial (15), FP64
FLOPS_PER_SEGMENT = 135        # winner's hit record (75) + shade (~60), FP64
# Algorithmic HBM bytes per segment (ray 48 + throughput 24 + id 4, read once and written once) and per path
# (float4 radiance write + read; float4 accumulate + f64 frame write per pixel)
BYTES_PER_SEGMENT = 2 * 76
ISSUE_PEAK = 4 * 32            # thread-instructions per cycle per SM: 4 schedulers x 32 lanes


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (profiling recipe)."""

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.gpu_index = gpu_index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                smax = float(r[1])
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# the reference arm / cpu_baseline: the oracle alone (never the product package)
# ------------------------------------------------------------------------------------------------
def cpu_sample_spp(cfg: str) -> int:
    """samples per pixel of the CPU arm's step: the WHOLE frame of the configuration (every pixel, the image's own
    mix of cheap and expensive regions) at the sample count that makes a step about 4 M paths; Mpaths/s does not
    depend on spp"""
    c = CONFIGS[cfg]
    return max(1, min(c["spp"], round(4.0e6 / (c["w"] * c["h"]))))


def cpu_reference_run(cfg: str, steps: int, warmup: int):
    """The reference's own CPU implementation of the path, as far as this image can run it: the oracle's threaded
    renderer (1 serial dispatcher + T workers, BVH as Scene::new builds it) on all host threads.  Loads
    oracle/scenes/cfg*.npz (written by tools/make_oracle_scenes.py); imports nothing of the product."""
    from oracle import pyoracle as po
    threads = po.hardware_threads()
    if cfg == "2":
        return cpu_rays_run(po, threads, steps, warmup)
    c = CONFIGS[cfg]
    osc, cam = po.load_flat_scene(os.path.join(ROOT, "oracle", "scenes", f"cfg{cfg}.npz"))
    osc.build_bvh(seed=1)
    spp = cpu_sample_spp(cfg)
    n_paths = c["w"] * c["h"] * spp
    secs, counters = [], None
    for i in range(warmup + steps):
        frame, info = osc.render(cam, c["w"], c["h"], spp, DEPTH, seed=RNG_SEED + i, rng="xoshiro", use_bvh=True,
                                 threads=threads, counters=(i == warmup + steps - 1))
        if i >= warmup:
            secs.append(info["seconds"])
        counters = info.get("counters", counters)
    mean_s = sum(secs) / len(secs)
    desc = (f"the whole {c['w']}x{c['h']} frame of the configuration at {spp} spp (of {c['spp']}), depth {DEPTH} = "
            f"{n_paths} paths per step; C++ restatement of the reference's threaded renderer with its BVH, {threads} "
            f"worker threads + 1 serial dispatcher (not the Rust binary: no Rust toolchain in the image)")
    return {"value": n_paths / mean_s / 1e6, "unit": "Mpaths/s", "ms": mean_s * 1e3, "cores": threads, "sample": desc,
            "n_units": n_paths, "counters": counters, "outputs": {"frame": frame}}


def bench_rays(n, seed=42, target_radius=3.0):
    """benches/bench_intersections.rs:69-70: origin = -random_in_sphere(10), direction toward a point jittered inside
    a ball around the origin (so that about half of the rays miss; SURVEY 8d cfg 2).  Directions normalised like
    Ray::new: d / sqrt((x*x + y*y) + z*z)."""
    import numpy as np
    rng = np.random.default_rng(seed)

    def ball(m, r):
        out = np.empty((0, 3))
        while out.shape[0] < m:
            v = rng.uniform(-r, r, (2 * m, 3))
            out = np.concatenate([out, v[(v * v).sum(1) <= r * r]])
        return out[:m]

    o = -ball(n, 10.0)
    d = ball(n, target_radius) - o
    d = d / np.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1] + d[:, 2] * d[:, 2])[:, None]
    return np.ascontiguousarray(np.concatenate([o, d], axis=1))


def cpu_rays_run(po, threads, steps, warmup):
    osc, _ = po.load_flat_scene(os.path.join(ROOT, "oracle", "scenes", "cfg2.npz"))
    rays = bench_rays(CONFIGS["2"]["rays"])
    secs = []
    for i in range(warmup + steps):
        out = osc.intersect_batch(rays, threads=threads)
        if i >= warmup:
            secs.append(out["seconds"])
    mean_s = sum(secs) / len(secs)
    return {"value": len(rays) / mean_s / 1e6, "unit": "Mrays/s", "ms": mean_s * 1e3, "cores": threads,
            "sample": f"all {len(rays)} rays per step, ShapeCollection loop (no BVH), {threads} threads; C++ restatement "
                      "of the reference (not the Rust binary)", "n_units": len(rays), "counters": None,
            "outputs": {k: out[k] for k in ("index", "t", "normal")}}


DUMP_LIMIT = 64_000_000    # bytes --dump-outputs writes at most
DUMP_SEED = 20240601


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """--dump-outputs: every array as out_dir/<name>.npy in float64 (shape indices are exact in it).  The arrays share
    their first axis (image rows, rays); when together they exceed DUMP_LIMIT, the same fixed, seeded sample of that
    axis is kept from each, in increasing order, and its indices are written as out_dir/sample_index.npy."""
    import numpy as np
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    n = len(next(iter(arrays.values())))
    per_item = sum(a.nbytes for a in arrays.values()) // n
    if n * per_item > DUMP_LIMIT:
        keep = (DUMP_LIMIT - 4096) // (per_item + 8)      # (+ the index array, + the .npy headers)
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(n, keep, replace=False))
        arrays = {k: a[idx] for k, a in arrays.items()}
        arrays["sample_index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def emit(line: dict) -> None:
    """the ONE JSON line, on the real stdout"""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1


def ncu_kernels():
    """profiles/ncu_kernels.json: per-kernel issue-slot utilisation and active lanes from the committed
    `ncu --set full` capture of this build (tools/ncu_kernels_json.py); None when absent"""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "ncu_kernels.json")))
    except Exception:
        return None


def lane_weighted_issue(entry):
    """duration-weighted over the captured launches: issue-slot utilisation x active lanes / 32"""
    tot = sum(l["duration_us"] for l in entry["launches"])
    return {
        "issue_slot_frac": sum(l["issue_slot_pct"] / 100.0 * l["duration_us"] for l in entry["launches"]) / tot,
        "active_lanes_of_32": sum(l["active_lanes"] * l["duration_us"] for l in entry["launches"]) / tot,
        "lane_weighted_issue_frac": sum(l["issue_slot_pct"] / 100.0 * l["active_lanes"] / 32.0 * l["duration_us"]
                                        for l in entry["launches"]) / tot,
        "fp64_pipe_frac": sum(l.get("fp64_pipe_pct", 0.0) / 100.0 * l["duration_us"] for l in entry["launches"]) / tot,
        "dram_bytes_per_launch": [l.get("dram_bytes") for l in entry["launches"]],
    }


def main():
    # libraries (NCCL's version banner, torch warnings) must not share stdout with the JSON line: keep a
    # private duplicate of fd 1 for it and point fd 1 at stderr for everybody else
    global _REAL_STDOUT
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="3", choices=sorted(CONFIGS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")

    in_torchrun = "WORLD_SIZE" in os.environ
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "ours" and not in_torchrun and args.gpus > 1:
        # `python bench.py --gpus N`: one process per GPU needs a launcher -- re-launch under torchrun
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", os.environ.get("MASTER_PORT", "29517"),
               os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd)
    if args.impl == "ours" and in_torchrun and args.gpus != world:
        raise SystemExit(f"bench.py: --gpus {args.gpus} but the launcher started {world} rank(s)")

    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cfg = args.config
    C_ = CONFIGS[cfg]
    unit = "Mrays/s" if cfg == "2" else "Mpaths/s"
    config = {"workload": C_["workload"], "config": cfg, "scene_seed": SCENE_SEED,
              "parallelism": (f"contiguous ray ranges over {world} GPU(s), no exchange" if cfg == "2" else
                              f"interleaved 32x32 tiles over {world} GPU(s); the K timed steps run as one pipelined "
                              "sequence of complete frames (step n's exchange / assembly / host copy overlap step n+1's render)"),
              "l2_policy": ("1 Mi rays in (48 MB) + hit records out (60 MB) per step exceed nothing: L2 flushed by a 256 MB "
                            "write between steps" if cfg == "2" else
                            "per-step queues (>= 1.9 GB of path state streamed per batch) exceed the 126 MB L2; no explicit flush")}

    if args.impl == "reference":
        if rank != 0:
            return 0
        assert "rs_pathtracing_b200" not in sys.modules
        r = cpu_reference_run(cfg, args.steps, args.warmup)
        assert "rs_pathtracing_b200" not in sys.modules   # the reference arm runs the oracle alone
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, r["outputs"])
        line = {"impl": "reference", "metric": unit, "value": r["value"], "unit": unit, "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms"], "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": r["value"], "unit": unit, "cores": r["cores"], "kind": "port",
                                 "sample": r["sample"]},
                "e2e": {"value": r["value"], "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        emit(line)
        return 0

    import numpy as np
    import torch
    import rs_pathtracing_b200 as rt

    if not torch.cuda.is_available() or rt.device_count() == 0:
        raise SystemExit("bench.py needs a CUDA device: the core has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    def sum_over_ranks(x: float) -> float:
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t[0])

    ctx = dict(args=args, rank=rank, world=world, local_rank=local_rank, dist=dist, barrier=barrier,
               max_over_ranks=max_over_ranks, sum_over_ranks=sum_over_ranks, config=config, unit=unit)
    line = run_rays(ctx) if cfg == "2" else run_frames(ctx, cfg)
    if rank == 0 and line is not None:
        emit(line)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def load_config_scene(cfg):
    import numpy as np
    import rs_pathtracing_b200 as rt
    sc = rt.Scene.from_file(os.path.join(ROOT, "scenes", CONFIGS[cfg]["scene"]), random_spheres_seed=SCENE_SEED)
    cam = sc.camera()
    if cfg == "4b":
        sc.assign_material(1, "EarthMap")        # Sphere1  -> Metal + ImageTexture
        sc.assign_material(2, "Glass")           # Cushion  -> Dielectric
        sc.assign_material(5, "Lambertian01")    # a random sphere -> Lambertian + UVChecker
        sc.assign_material(6, "WhiteMirror")
        pos = np.array(cam.position.tuple())
        cam = rt.camera_new(pos, -pos, (0, 1, 0), 1.0, cam.fov_rad)
    return sc, cam


def run_frames(ctx, cfg):
    import ctypes as C
    import numpy as np
    import torch
    import rs_pathtracing_b200 as rt
    from rs_pathtracing_b200 import api, _ffi
    from rs_pathtracing_b200.distributed import DistributedRenderer

    args, rank, world, local_rank = ctx["args"], ctx["rank"], ctx["world"], ctx["local_rank"]
    barrier, max_over_ranks, sum_over_ranks = ctx["barrier"], ctx["max_over_ranks"], ctx["sum_over_ranks"]
    C_ = CONFIGS[cfg]
    WIDTH, HEIGHT, SPP = C_["w"], C_["h"], C_["spp"]

    t_up0 = time.perf_counter()
    sc, cam = load_config_scene(cfg)
    dr = DistributedRenderer(sc, DEPTH, seed=RNG_SEED, tile=32, device=local_rank)
    scene_upload_ms = (time.perf_counter() - t_up0) * 1e3
    n_paths = WIDTH * HEIGHT * SPP

    # --- kernel-side measurement: device-resident inputs, frame left on the device ---------------
    dr.render_many_device(cam, WIDTH, HEIGHT, SPP, args.warmup)   # (the warm-up steps through the same pipelined path)
    barrier()
    sc.reset_stats(local_rank)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    frame_ms = []
    barrier()
    t0 = time.perf_counter()
    # the K steps as ONE pipelined sequence: every step renders and assembles a complete frame; step n's exchange to
    # rank 0 and its k_assemble overlap step n+1's render (DistributedRenderer.render_jobs_device)
    last_frame = dr.render_many_device(cam, WIDTH, HEIGHT, SPP, args.steps,
                                       on_rendered=lambda i: frame_ms.append(sc.stats(local_rank).last_frame_ms))   # CUDA events on the library's stream
    barrier()
    wall_s = time.perf_counter() - t0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:   # (the passes below reuse the frame buffer)
        dump_outputs(args.dump_outputs, {"frame": last_frame.cpu().numpy()})
    launches = sc.stats(local_rank).kernel_launches
    # per-kernel device time: the same K steps again with one CUDA event pair around every launch on the
    # library's stream (the event pairs serialise the two stream lanes, so they stay out of the pass `value` comes from)
    sc.set_kernel_timing(True, local_rank)
    sc.reset_stats(local_rank)
    timed_ms = []
    for _ in range(args.steps):
        dr.render_device(cam, WIDTH, HEIGHT, SPP)
        timed_ms.append(sc.stats(local_rank).last_frame_ms)
    barrier()
    kst = sc.stats(local_rank)
    kernel_ms = {"k_raygen": kst.ms_raygen / args.steps, "k_extend": kst.ms_extend / args.steps,
                 "k_march": kst.ms_march / args.steps, "k_shade": kst.ms_shade / args.steps,
                 "k_resolve": kst.ms_resolve / args.steps}
    kernel_launches = {"k_extend": kst.launches_extend / args.steps, "k_march": kst.launches_march / args.steps,
                       "k_shade": kst.launches_shade / args.steps}
    sc.set_kernel_timing(False, local_rank)
    step_ms = max_over_ranks(wall_s * 1e3 / args.steps)
    launches = int(sum_over_ranks(float(launches)))
    value = n_paths / (step_ms * 1e-3) / 1e6

    # --- end to end through the public API: host buffers, D2H inside the timed region ------------
    host_frame = dr.render_jobs([(cam, WIDTH, HEIGHT, SPP)] * 2)   # (warm-up: pinned host buffers)
    barrier()
    t0 = time.perf_counter()
    host_frame = dr.render_jobs([(cam, WIDTH, HEIGHT, SPP)] * args.steps)   # every frame lands in pinned host memory
    barrier()
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3 / args.steps)
    e2e_value = n_paths / (e2e_ms * 1e-3) / 1e6
    h2d = C.sizeof(_ffi.Camera) + C.sizeof(_ffi.RenderParams)
    d2h = WIDTH * HEIGHT * 24

    # --- frame check (untimed): consecutive bench frames are identical, which would hide a frame assembled from
    # stale shard buffers; so one more frame with ANOTHER seed and fewer samples goes through the same
    # DistributedRenderer and is compared, on rank 0, with the unsharded render of that seed -----------------
    frame_check = None
    try:
        dr.seed = RNG_SEED + 1
        check_spp = min(16, SPP)
        chk = dr.render(cam, WIDTH, HEIGHT, check_spp)        # collective: every rank takes part
        dr.seed = RNG_SEED
        if rank == 0:
            sc2, _ = load_config_scene(cfg)
            ref = np.full((HEIGHT, WIDTH, 3), -1.0)
            d2 = sc2.device_scene(local_rank)
            api.render_start(d2, cam, api.render_params(WIDTH, HEIGHT, check_spp, DEPTH, RNG_SEED + 1))
            api.render_wait(d2, ref)
            # the exchanged accumulators hold float sums: equal to the f64 frame up to float rounding
            bad = (np.abs(chk - ref) > 3e-7 * np.maximum(np.abs(ref), 1e-9)).any(axis=2)
            frame_check = {"what": f"DistributedRenderer frame (seed {RNG_SEED + 1}, {check_spp} spp) against the unsharded "
                                   "render on rank 0, tolerance 3e-7 relative", "deviating_pixels": int(bad.sum())}
    except Exception as e:   # the check must never cost the bench line
        frame_check = {"error": repr(e)}
    barrier()

    if rank != 0:
        return None
    assert host_frame is not None and np.isfinite(host_frame).all() and host_frame.mean() > 0.01
    # --- work counters of rank 0's shard: one instrumented frame at reduced spp (counts scale linearly with spp) ----
    count_spp = min(4, SPP)
    sc.set_counters(True, local_rank)
    sc.reset_stats(local_rank)
    p = api.render_params(WIDTH, HEIGHT, count_spp, DEPTH, RNG_SEED, world, 0, tile=32)
    api.render_start(dr.dev_scene, cam, p)
    api.render_wait(dr.dev_scene, None)
    st = sc.stats(local_rank)
    sc.set_counters(False, local_rank)
    scale = SPP / count_spp
    segs, exact, culls, evals, mrays = (st.segments * scale, st.shape_tests * scale, st.cull_tests * scale,
                                        st.march_steps * scale, st.march_rays * scale)
    n_shapes = sc.shape_count
    shard_paths = n_paths / world
    shard_ms = sum(timed_ms) / len(timed_ms)   # the single-lane pass the per-kernel times come from
    fp64_peak, fp32_peak = rt.measure_peaks(local_rank)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        r = cpu_reference_run(cfg, steps=1, warmup=0)
        cpu = {"value": r["value"], "unit": "Mpaths/s", "cores": r["cores"], "kind": "port", "sample": r["sample"],
               "ms": r["ms"], "counters_per_path": {k: v / r["n_units"] for k, v in (r["counters"] or {}).items()}}

    # --- roofline: the kernel with the largest share of the step ------------------------------------------------
    ncu = ncu_kernels()
    executed = {   # executed arithmetic per kernel class, from the live counters (FP64 unless noted)
        "k_extend": {"fp64_flops": exact * FLOPS_PER_SHAPE_TEST, "fp32_flops": culls * FLOPS_PER_CULL_TEST},
        "k_march": {"fp64_flops": evals * FLOPS_PER_MARCH_STEP, "fp32_flops": 0.0},
        "k_shade": {"fp64_flops": segs * FLOPS_PER_SEGMENT, "fp32_flops": 0.0},
    }
    kernels = {}
    for name, ms in kernel_ms.items():
        k = {"ms_per_step": ms, "share_of_step": ms / shard_ms}
        if name in kernel_launches:
            k["launches_per_step"] = kernel_launches[name]
            k["ms_per_launch"] = ms / max(kernel_launches[name], 1)
        if name in executed and ms > 0:
            k["executed_fp64_tflops"] = executed[name]["fp64_flops"] / (ms * 1e-3) / 1e12
            k["executed_fp64_frac_of_dfma_peak"] = k["executed_fp64_tflops"] / fp64_peak
            if executed[name]["fp32_flops"]:
                k["executed_fp32_tflops"] = executed[name]["fp32_flops"] / (ms * 1e-3) / 1e12
                k["executed_fp32_frac_of_ffma_peak"] = k["executed_fp32_tflops"] / fp32_peak
        if ncu and name in ncu.get("kernels", {}):
            k["ncu"] = lane_weighted_issue(ncu["kernels"][name])
        kernels[name] = k
    dominant = max(kernel_ms, key=kernel_ms.get)
    dom = kernels[dominant]
    issue = dom.get("ncu", {}).get("lane_weighted_issue_frac")
    # algorithmic work of the reference's formulation (what its CPU path executes for the same frame): every shape
    # tested for every segment + every literal marching step (oracle counters, per path, from the cpu_baseline leg's
    # BVH-free definition: segments x shapes x 52; literal march steps x 22) -- reported as a ratio to the executed
    # work, never as a utilisation
    literal_steps_per_path = (cpu or {}).get("counters_per_path", {}).get("march_steps")
    alg_flops = segs * n_shapes * FLOPS_PER_SHAPE_TEST + segs * FLOPS_PER_SEGMENT
    if literal_steps_per_path is not None:
        alg_flops += literal_steps_per_path * shard_paths * FLOPS_PER_MARCH_STEP
    exe_flops = sum(v["fp64_flops"] + v["fp32_flops"] for v in executed.values())
    hbm_bytes = segs * BYTES_PER_SEGMENT + shard_paths * 32 + (WIDTH * HEIGHT / world) * 40
    hbm_gbs = hbm_bytes / (shard_ms * 1e-3) / 1e9
    roofline = {
        "bound": "issue (FP64 reference arithmetic, divergent control flow; no dense contraction, tensor cores unused)",
        "kernel": dominant,
        "achieved": None if issue is None else issue * ISSUE_PEAK, "peak": ISSUE_PEAK,
        "unit": "thread-instructions / cycle / SM", "frac": issue,
        "frac_is": "SM issue-slot utilisation x active lanes / 32 of the dominant kernel, duration-weighted over the "
                   "launches of the committed ncu --set full capture of this build (profiles/ncu_kernels.json: "
                   + (ncu or {}).get("capture", "absent") + "); peak = 4 schedulers x 32 lanes",
        "kernel_ms_per_step": dom["ms_per_step"], "share_of_step": dom["share_of_step"],
        "kernels": kernels,
        "fp_peaks": {"fp64_dfma_tflops": fp64_peak, "fp32_ffma_tflops": fp32_peak,
                     "source": "rt_measure_peaks: FMA micro-kernels timed live on this GPU (FMA = 2 flop); the bit-exact "
                               "contract forbids FMA contraction, so reference arithmetic tops out at 0.5 of them"},
        "work_per_step": {"segments": segs, "shapes": n_shapes, "exact_tests_per_segment": exact / max(segs, 1),
                          "pretests_per_segment": culls / max(segs, 1), "marched_rays": mrays,
                          "surface_evaluations": evals, "evaluations_per_marched_ray": evals / max(mrays, 1),
                          "literal_march_steps_per_path_reference": literal_steps_per_path},
        "algorithmic_speedup": {"reference_formulation_flops_per_step": alg_flops, "executed_flops_per_step": exe_flops,
                                "ratio": alg_flops / max(exe_flops, 1.0),
                                "note": "work the cull tree and exact-skip marching avoid; not a utilisation figure"},
        "flops_model": {"per_shape_test": FLOPS_PER_SHAPE_TEST, "per_pretest_fp32": FLOPS_PER_CULL_TEST,
                        "per_march_step": FLOPS_PER_MARCH_STEP, "per_segment": FLOPS_PER_SEGMENT},
        "traffic": (dom.get("ncu", {}).get("dram_bytes_per_launch") or [None])[0],
        "hbm": {"achieved": hbm_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_gbs / hbm_peak,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6650",
                "algorithmic_bytes_per_step": hbm_bytes},
    }
    return {
        "metric": "Mpaths/s", "value": value, "unit": "Mpaths/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": ctx["config"],
        "device_ms_per_step_rank0": sum(frame_ms) / len(frame_ms),
        "e2e": {"value": e2e_value, "unit": "Mpaths/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "scene_upload_ms_once": scene_upload_ms},
        "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
        "frame_check": frame_check,
    }


def run_rays(ctx):
    """config 2: rt_intersect_batch (RT_ISECT_FAST) on 1 Mi rays, contiguous ray ranges per rank, no exchange"""
    import ctypes as C
    import numpy as np
    import torch
    import rs_pathtracing_b200 as rt
    from rs_pathtracing_b200 import _ffi

    args, rank, world, local_rank = ctx["args"], ctx["rank"], ctx["world"], ctx["local_rank"]
    barrier, max_over_ranks = ctx["barrier"], ctx["max_over_ranks"]
    sc = rt.Scene.from_json(json.dumps(TRIO_SCENE), add_random_spheres=False)
    rays_all = bench_rays(CONFIGS["2"]["rays"])
    n_all = len(rays_all)
    lo, hi = rank * n_all // world, (rank + 1) * n_all // world
    rays = rays_all[lo:hi]
    n = len(rays)
    ds = sc.device_scene(local_rank)
    dev = f"cuda:{local_rank}"
    d_rays = torch.from_numpy(rays).to(dev)
    d_idx = torch.empty(n, dtype=torch.int32, device=dev)
    d_t = torch.empty(n, dtype=torch.float64, device=dev)
    d_n = torch.empty((n, 3), dtype=torch.float64, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream().cuda_stream or 0x1   # 0x1 = cudaStreamLegacy (0 would mean the library's stream)
    core = _ffi.core()

    def launch():
        rc = core.rt_intersect_batch_device(ds, d_rays.data_ptr(), n, 0.001, float("inf"), rt.RT_ISECT_FAST, d_idx.data_ptr(),
                                            d_t.data_ptr(), d_n.data_ptr(), None, None, None, C.c_void_p(stream))
        assert rc == 0, core.rt_last_error()

    for _ in range(args.warmup):
        flush.zero_()
        launch()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    evs = []
    for _ in range(args.steps):
        flush.zero_()                                   # L2 flush between timed iterations (not timed)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        launch()
        b.record()
        evs.append((a, b))
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:   # rank 0's rays
        dump_outputs(args.dump_outputs, {"index": d_idx.cpu().numpy(), "t": d_t.cpu().numpy(), "normal": d_n.cpu().numpy()})
    ms = max_over_ranks(sum(a.elapsed_time(b) for a, b in evs) / args.steps)
    value = n_all / (ms * 1e-3) / 1e6
    # end to end: host rays in, host hit records out through rt_intersect_batch
    sc.closest_hit(rays, mode=rt.RT_ISECT_FAST, device=local_rank, want=("index", "t", "normal"))
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = sc.closest_hit(rays, mode=rt.RT_ISECT_FAST, device=local_rank, want=("index", "t", "normal"))
    barrier()
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3 / args.steps)
    if rank != 0:
        return None
    assert np.array_equal(out["index"], d_idx.cpu().numpy())
    hit = out["index"] >= 0
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        r = cpu_reference_run("2", steps=1, warmup=0)
        cpu = {"value": r["value"], "unit": "Mrays/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]}
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    bytes_step = n * (48 + 4 + 8 + 24)
    gbs = bytes_step / (ms * 1e-3) / 1e9
    ncu = ncu_kernels()
    k = (ncu or {}).get("kernels", {}).get("k_intersect_batch")
    issue = lane_weighted_issue(k) if k else None
    return {"metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": ctx["config"], "hit_fraction": float(hit.mean()),
            "e2e": {"value": n_all / (e2e_ms * 1e-3) / 1e6, "unit": "Mrays/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": n * 48, "d2h_bytes_per_step": n * (4 + 8 + 24)},
            "gpu_launches": args.steps + args.warmup + args.steps + 1, "clocks": clocks,
            "roofline": {"bound": "issue (FP64 reference arithmetic + marching)", "kernel": "k_intersect_batch",
                         "achieved": None if issue is None else issue["lane_weighted_issue_frac"] * ISSUE_PEAK,
                         "peak": ISSUE_PEAK, "unit": "thread-instructions / cycle / SM",
                         "frac": None if issue is None else issue["lane_weighted_issue_frac"], "ncu": issue, "traffic": None,
                         "hbm": {"achieved": gbs, "peak": peaks.get("hbm_gbs", 6650.0), "unit": "GB/s",
                                 "frac": gbs / peaks.get("hbm_gbs", 6650.0), "algorithmic_bytes_per_step": bytes_step}},
            "cpu_baseline": cpu}


_IDENT = {"translate": [0, 0, 0], "rotate": [0, 0, 0], "scale": [1, 1, 1]}
TRIO_SCENE = {   # the shapes of benches/bench_intersections.rs:16-66
    "camera": {"position": [0, 0, -10], "direction": [0, 0, 1], "up": [0, 1, 0], "fov": 40.0, "focal_length": 1.0},
    "background": [0, 0, 0],
    "materials": {"M": {"type": "Lambertian", "albedo": {"type": "SolidColor", "color": [0.9, 0.1, 0.1]}}},
    "shapes": [{"type": "Sphere", "name": "Test sphere", "material": "M", "transform": _IDENT},
               {"type": "Cube", "name": "Test cube", "material": "M", "transform": _IDENT},
               {"type": "BruteForsableShape", "shape": {"type": "Heart"}, "step": 0.01, "material": "M", "transform": _IDENT}],
}


if __name__ == "__main__":
    sys.exit(main())
