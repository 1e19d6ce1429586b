"""The bins' render-and-save (src/bin/main_raylib.rs: RendererState::render + the 'S' key) without the window:

  python tools/render.py scenes/cornell_box.json out.png --size 1024 1024 --spp 256 [--depth 8] [--seed 1]
      [--adaptive REL [--min-samples N] [--abs-error A] [--heatmap counts.png]]
      [--counts MAP.npy [--heatmap counts.png]]
      [--orbit N] [--animate N [--step S]] [--inspect X Y] [--layers N] [--features]

With --layers N, the frame and its N bounce layers (rt_render_start_layers): layer b holds the light of the paths that
ended on bounce level b (the last layer: on level N-1 or deeper); layer b goes to OUT_Lb.png (out_L00.png, ... for
out.png), tone-mapped like the frame, and each layer's share of the frame's mean luminance is printed -- what depth is
enough for the scene.

With --features, the frame and the first-hit features of its samples' camera rays (rt_render_start_features), the inputs
a denoiser takes beside the colour: OUT_albedo.png (the hit's material colour, sky at a miss, clamped to [0, 1]),
OUT_normal.png (0.5 n + 0.5 of the mean world normal), OUT_depth.png (mean hit distance, near = white, normalised over
the finite values; no hit = black) and OUT_shape.png (a hashed colour per shape id of sample 0, miss = black); the mean
coverage (the share of samples that hit something) is printed.

Scene::from_json -> GpuRenderer (Renderer trait: start_rendering / render_step until done) ->
rt_tonemap_rgba8 (sqrt, clamp(0, 0.999) * 256, on the device) -> PNG.  With --adaptive, an adaptive frame
(rt_render_start_adaptive): every pixel gets --min-samples samples and doubles its count, up to --spp, while the
standard error of its mean luminance exceeds REL times the mean (or --abs-error); --heatmap writes the per-pixel
sample counts as a grey PNG (black = min-samples, white = spp, log2 scale).  With --counts, a frame with the given
sample count per pixel (rt_render_start_counts): MAP.npy is an (h, w) uint32 array, which sets the size; --heatmap
then draws that map (black = 0 or 1 sample, white = its largest count, log2 scale) and the frame's count-0 pixels
are black.  With --orbit N, one frame of N views (rt_render_start_views): the scene camera's position and direction
rotated about the world y axis through the origin by 360/N degrees at a time; view k goes to OUT_k.png (out_000.png,
out_001.png, ... for out.png).  With --animate N, N frames in which the scene's random spheres move on a seeded
random walk in the x-z plane (--step per axis and frame), each frame on the same renderer after
Scene.set_transforms-style edits of the scene (rt_scene_update_transforms: the cull tree is refit in place); frame k
goes to OUT_k.png.  With --inspect X Y, after the frame: every sample's path of pixel (X, Y), traced again level by
level with Scene.scatter (api.trace_paths on the frame's own primary rays, api.primary_rays): at each level the shape
and material hit, the outcome and the throughput, then the sample's radiance; the mean of the samples must be the
frame's pixel bit for bit."""
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
ap.add_argument("--counts", default=None, metavar="MAP.npy", help="(h, w) uint32 sample count per pixel")
ap.add_argument("--heatmap", default=None, help="PNG of the per-pixel sample counts (with --adaptive or --counts)")
ap.add_argument("--orbit", type=int, default=None, metavar="N", help="N views around the scene, one PNG per view")
ap.add_argument("--animate", type=int, default=None, metavar="N", help="N frames of the random spheres on a random walk")
ap.add_argument("--step", type=float, default=0.05, help="--animate: random-walk step per axis and frame")
ap.add_argument("--layers", type=int, default=None, metavar="N", help="N bounce layers, one PNG per layer")
ap.add_argument("--features", action="store_true", help="albedo, normal, depth and shape PNGs of the first hits")
ap.add_argument("--inspect", type=int, nargs=2, default=None, metavar=("X", "Y"),
                help="print each sample's path of pixel (X, Y) and check their mean against the frame")
a = ap.parse_args()
if a.inspect is not None and (a.orbit is not None or a.animate is not None or a.adaptive is not None
                              or a.counts is not None):
    ap.error("--inspect excludes --orbit, --animate, --adaptive and --counts")
if a.inspect is not None and not (0 <= a.inspect[0] < a.size[0] and 0 <= a.inspect[1] < a.size[1]):
    ap.error(f"--inspect: pixel {tuple(a.inspect)} outside the {a.size[0]}x{a.size[1]} image")
if a.orbit is not None and (a.orbit < 1 or a.adaptive is not None or a.counts is not None):
    ap.error("--orbit needs N >= 1 and excludes --adaptive and --counts")
if a.animate is not None and (a.animate < 1 or a.orbit is not None or a.adaptive is not None or a.counts is not None):
    ap.error("--animate needs N >= 1 and excludes --orbit, --adaptive and --counts")
if a.layers is not None and (not 1 <= a.layers <= 63 or a.orbit is not None or a.animate is not None
                             or a.adaptive is not None or a.counts is not None or a.inspect is not None):
    ap.error("--layers needs 1 <= N <= 63 and excludes --orbit, --animate, --adaptive, --counts and --inspect")
if a.features and (a.layers is not None or a.orbit is not None or a.animate is not None or a.adaptive is not None
                   or a.counts is not None or a.inspect is not None):
    ap.error("--features excludes --layers, --orbit, --animate, --adaptive, --counts and --inspect")
if a.heatmap and a.adaptive is None and a.counts is None:
    ap.error("--heatmap needs --adaptive or --counts")
if a.adaptive is not None and a.counts is not None:
    ap.error("--adaptive and --counts exclude each other")
sc = rt.Scene.from_file(a.scene, random_spheres_seed=a.seed)
cam = sc.camera()
r = rt.GpuRenderer(sc, 12, a.depth, seed=a.seed)
w, h = a.size
if a.counts is not None:
    given = np.load(a.counts)
    if given.ndim != 2 or given.dtype != np.uint32:
        ap.error(f"--counts: an (h, w) uint32 array expected, got {given.dtype} {given.shape}")
    h, w = given.shape
t0 = time.perf_counter()
if a.layers is not None:
    frame, layers = r.render_layers(cam, w, h, a.spp, a.layers)
    dt = time.perf_counter() - t0
    stem, ext = os.path.splitext(a.out)
    rt.save_png(a.out, rt.tonemap_rgba8(sc, frame))
    y = lambda f: float(np.mean((0.2126 * f[..., 0] + 0.7152 * f[..., 1]) + 0.0722 * f[..., 2]))
    total = y(frame)
    print(f"{a.scene}: {w}x{h}x{a.spp}, depth {a.depth}, {a.layers} layers in {dt * 1e3:.1f} ms -> {a.out}")
    for b in range(a.layers):
        rt.save_png(f"{stem}_L{b:02d}{ext or '.png'}", rt.tonemap_rgba8(sc, layers[b]))
        share = y(layers[b]) / total if total else 0.0
        last = "+" if b == a.layers - 1 and a.layers <= a.depth else " "
        print(f"  level {b:2d}{last} {100.0 * share:8.4f} % of the mean luminance  -> {stem}_L{b:02d}{ext or '.png'}")
    sys.exit(0)
if a.features:
    frame, f = r.render_features(cam, w, h, a.spp)
    dt = time.perf_counter() - t0
    stem, ext = os.path.splitext(a.out)
    rt.save_png(a.out, rt.tonemap_rgba8(sc, frame))
    rgba = lambda c: np.concatenate([np.clip(np.nan_to_num(c) * 255.0 + 0.5, 0, 255).astype(np.uint8),
                                     np.full(c.shape[:2] + (1,), 255, np.uint8)], axis=2)
    d = f["depth"]
    finite = np.isfinite(d)
    lo, hi = (float(d[finite].min()), float(d[finite].max())) if finite.any() else (0.0, 1.0)
    near = np.where(finite, 1.0 - (d - lo) / (hi - lo if hi > lo else 1.0), 0.0)
    ids = f["shape"].astype(np.uint32)
    hashed = [((ids * np.uint32(0x9E3779B1)) >> np.uint32(s)) & np.uint32(255) for s in (8, 16, 24)]
    shape_rgb = np.where((f["shape"] >= 0)[..., None], np.stack(hashed, 2) / 255.0, 0.0)
    outs = {"albedo": f["albedo"], "normal": 0.5 * f["normal"] + 0.5, "depth": np.repeat(near[..., None], 3, 2),
            "shape": shape_rgb}
    print(f"{a.scene}: {w}x{h}x{a.spp}, depth {a.depth}, features in {dt * 1e3:.1f} ms -> {a.out}; "
          f"coverage {100.0 * float(f['coverage'].mean()):.4f} % of the samples hit a shape")
    for k, img in outs.items():
        path = f"{stem}_{k}{ext or '.png'}"
        rt.save_png(path, rgba(img))
        print(f"  {k:6s} -> {path}")
    sys.exit(0)
if a.orbit is not None:
    views = r.render_views(rt.api.orbit_cameras(cam, a.orbit), w, h, a.spp)
    dt = time.perf_counter() - t0
    stem, ext = os.path.splitext(a.out)
    for k in range(a.orbit):
        rt.save_png(f"{stem}_{k:03d}{ext or '.png'}", rt.tonemap_rgba8(sc, views[k]))
    paths = a.orbit * w * h * a.spp
    print(f"{a.scene}: {a.orbit} views of {w}x{h}x{a.spp} in {dt * 1e3:.1f} ms ({paths / dt / 1e6:.1f} Mpaths/s) "
          f"-> {stem}_000{ext or '.png'} .. {stem}_{a.orbit - 1:03d}{ext or '.png'}")
    sys.exit(0)
if a.animate is not None:
    n_file = rt.Scene.from_file(a.scene, add_random_spheres=False).shape_count
    walk = rt.api.random_walk(sc, np.arange(n_file, sc.shape_count), a.animate, a.step, seed=a.seed)
    stem, ext = os.path.splitext(a.out)
    for k, (index, inverse, direct) in enumerate(walk):
        sc.set_transform_rows(index, inverse, direct)   # the scene and the renderer's handle move together
        rt.save_png(f"{stem}_{k:03d}{ext or '.png'}", rt.tonemap_rgba8(sc, r.render(cam, w, h, a.spp)))
    dt = time.perf_counter() - t0
    print(f"{a.scene}: {a.animate} frames of {w}x{h}x{a.spp}, {sc.shape_count - n_file} spheres moving, in "
          f"{dt * 1e3:.1f} ms -> {stem}_000{ext or '.png'} .. {stem}_{a.animate - 1:03d}{ext or '.png'}")
    sys.exit(0)
if a.counts is not None:
    buf = r.render_counts(cam, given)
    counts = given
    paths = int(given.sum(dtype=np.uint64))
elif a.adaptive is None:
    buf = np.zeros((h, w, 3))
    r.start_rendering(cam, rt.ImageParams(w, h), a.spp)
    while not r.render_step(buf):
        time.sleep(0.001)
    paths = w * h * a.spp
else:
    buf, counts, _ = r.render_adaptive(cam, w, h, a.spp, min(a.min_samples, a.spp), a.adaptive, a.abs_error)
    paths = int(counts.sum())
dt = time.perf_counter() - t0
rt.save_png(a.out, rt.tonemap_rgba8(sc, buf))   # (a count-0 pixel is NaN, which the tone map makes black)
print(f"{a.scene}: {w}x{h}, {paths / (w * h):.1f} spp on average, in {dt * 1e3:.1f} ms "
      f"({paths / dt / 1e6:.1f} Mpaths/s) -> {a.out}")
if a.heatmap:
    if a.counts is not None:
        lo, hi = 0.0, np.log2(max(int(counts.max()), 1))
    else:
        lo, hi = np.log2(min(a.min_samples, a.spp)), np.log2(a.spp)
    with np.errstate(divide="ignore"):   # log2(0) = -inf: black
        level = (np.log2(counts.astype(np.float64)) - lo) / max(hi - lo, 1e-9)
    grey = np.round(np.clip(level, 0.0, 1.0) * 255).astype(np.uint8)
    rgba = np.dstack([grey, grey, grey, np.full_like(grey, 255)])
    rt.save_png(a.heatmap, rgba)
    print(f"sample counts: {dict(zip(*[v.tolist() for v in np.unique(counts, return_counts=True)]))} -> {a.heatmap}")
if a.inspect is not None:
    x, y = a.inspect
    rays, keys = rt.api.primary_rays(cam, w, h, [x + y * w], a.spp, a.seed)
    radiance, levels = rt.trace_paths(sc, rays, keys, a.depth, a.seed, record=True)
    d = sc.desc()
    kinds = ("Lambertian", "Metal", "Dielectric", "DiffuseLight", "EmptyMaterial")
    outcome = {rt.RT_BOUNCE_MISS: "miss (sky)", rt.RT_BOUNCE_SCATTER: "scatter", rt.RT_BOUNCE_EMIT: "emit"}
    for s in range(a.spp):
        print(f"pixel ({x}, {y}) sample {s}:")
        for level, v in enumerate(levels):
            at = np.flatnonzero(v["ray"] == s)
            if at.size == 0:
                break
            k = int(at[0])
            i, oc = int(v["shape"][k]), int(v["outcome"][k])
            col, beta = v["color"][k], v["beta"][k]
            what = "-" if i < 0 else f"{sc.shape_name(i)} ({kinds[d.materials[d.material[i]].kind]})"
            if oc != rt.RT_BOUNCE_MISS and level == a.depth:
                tag = "hit on the last level: black"
            else:
                tag = outcome[oc]
            after = beta * col if oc == rt.RT_BOUNCE_SCATTER and level < a.depth else beta
            print(f"  level {level:2d}: {what:40s} {tag:28s} colour {np.round(col, 4).tolist()}  "
                  f"throughput {np.round(after, 4).tolist()}")
        print(f"  radiance {radiance[s].tolist()}")
    mean = rt.group_means(radiance, [0, a.spp])[0]
    got = buf[y, x]
    print(f"pixel ({x}, {y}): mean of the {a.spp} paths {mean.tolist()}, frame {got.tolist()} -> "
          f"{'bit for bit' if np.array_equal(mean, got) else 'DIFFERENT'}")
    if not np.array_equal(mean, got):
        sys.exit(1)
