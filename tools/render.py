"""The bins' render-and-save (src/bin/main_raylib.rs: RendererState::render + the 'S' key) without the window:

  python tools/render.py scenes/cornell_box.json out.png --size 1024 1024 --spp 256 [--depth 8] [--seed 1]
      [--adaptive REL [--min-samples N] [--abs-error A] [--heatmap counts.png]]

Scene::from_json -> GpuRenderer (Renderer trait: start_rendering / render_step until done) ->
rt_tonemap_rgba8 (sqrt, clamp(0, 0.999) * 256, on the device) -> PNG.  With --adaptive, an adaptive frame
(rt_render_start_adaptive): every pixel gets --min-samples samples and doubles its count, up to --spp, while the
standard error of its mean luminance exceeds REL times the mean (or --abs-error); --heatmap writes the per-pixel
sample counts as a grey PNG (black = min-samples, white = spp, log2 scale)."""
import argparse, os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import rs_pathtracing_b200 as rt

ap = argparse.ArgumentParser()
ap.add_argument("scene")
ap.add_argument("out")
ap.add_argument("--size", type=int, nargs=2, default=[640, 480])
ap.add_argument("--spp", type=int, default=64)
ap.add_argument("--depth", type=int, default=50)   # the bins construct their renderer with depth 50
ap.add_argument("--seed", type=int, default=1)
ap.add_argument("--adaptive", type=float, default=None, metavar="REL", help="relative standard-error target")
ap.add_argument("--min-samples", type=int, default=8)
ap.add_argument("--abs-error", type=float, default=0.0)
ap.add_argument("--heatmap", default=None, help="PNG of the per-pixel sample counts (with --adaptive)")
a = ap.parse_args()
if a.heatmap and a.adaptive is None:
    ap.error("--heatmap needs --adaptive")
sc = rt.Scene.from_file(a.scene, random_spheres_seed=a.seed)
cam = sc.camera()
r = rt.GpuRenderer(sc, 12, a.depth, seed=a.seed)
w, h = a.size
t0 = time.perf_counter()
if a.adaptive is None:
    buf = np.zeros((h, w, 3))
    r.start_rendering(cam, rt.ImageParams(w, h), a.spp)
    while not r.render_step(buf):
        time.sleep(0.001)
    paths = w * h * a.spp
else:
    buf, counts, _ = r.render_adaptive(cam, w, h, a.spp, min(a.min_samples, a.spp), a.adaptive, a.abs_error)
    paths = int(counts.sum())
dt = time.perf_counter() - t0
rt.save_png(a.out, rt.tonemap_rgba8(sc, buf))
print(f"{a.scene}: {w}x{h}, {paths / (w * h):.1f} spp on average, in {dt * 1e3:.1f} ms "
      f"({paths / dt / 1e6:.1f} Mpaths/s) -> {a.out}")
if a.heatmap:
    lo, hi = np.log2(min(a.min_samples, a.spp)), np.log2(a.spp)
    level = (np.log2(counts.astype(np.float64)) - lo) / max(hi - lo, 1e-9)
    grey = np.round(np.clip(level, 0.0, 1.0) * 255).astype(np.uint8)
    rgba = np.dstack([grey, grey, grey, np.full_like(grey, 255)])
    rt.save_png(a.heatmap, rgba)
    print(f"sample counts: {dict(zip(*[v.tolist() for v in np.unique(counts, return_counts=True)]))} -> {a.heatmap}")
