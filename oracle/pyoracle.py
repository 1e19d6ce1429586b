"""ORACLE — TEST INFRASTRUCTURE ONLY.  ctypes loader for oracle/liboracle.so.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import
this module; the product package never does.  The scene description structs are the C-ABI types of
include/rt_b200.h (plain data, no code): when the product package is already imported (the tests) its
ctypes classes are used, so that structures pass between the two without conversion; otherwise (bench.py
--impl reference) the oracle's own copy in abi_types.py, and nothing of the product is loaded.
"""
from __future__ import annotations

import ctypes as C
import math
import os
import subprocess

import numpy as np

import sys

if "rs_pathtracing_b200" in sys.modules:
    from rs_pathtracing_b200._ffi import Camera, Image, ImageParams, Material, Perlin, Ray, SceneDesc, Texture, Vec3
else:
    from .abi_types import Camera, Image, ImageParams, Material, Perlin, Ray, SceneDesc, Texture, Vec3

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "liboracle.so")


def build(force: bool = False) -> str:
    srcs = [os.path.join(HERE, f) for f in ("oracle.cpp", "oracle_c.cpp", "oracle.hpp", "Makefile")]
    stale = force or not os.path.exists(SO) or any(os.path.getmtime(s) > os.path.getmtime(SO) for s in srcs)
    if stale:
        subprocess.run(["make", "-C", HERE, "-B" if force else "-s", "liboracle.so"], check=True,
                       capture_output=True)
    return SO


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO):
        build()
    L = C.CDLL(SO)
    d16 = C.POINTER(C.c_double)
    L.orc_mat_mul.argtypes = [d16, d16, d16]
    L.orc_mat_rotate.argtypes = [Vec3, d16]
    L.orc_transform_new.argtypes = [Vec3, Vec3, Vec3, d16, d16]
    for f in ("orc_transform_point", "orc_transform_vector", "orc_transform_normal"):
        getattr(L, f).argtypes = [d16, Vec3]
        getattr(L, f).restype = Vec3
    L.orc_aabb_transform.argtypes = [Vec3, Vec3, d16, C.POINTER(Vec3), C.POINTER(Vec3)]
    L.orc_reflect.argtypes = [Vec3, Vec3]
    L.orc_reflect.restype = Vec3
    L.orc_refract.argtypes = [Vec3, Vec3, C.c_double]
    L.orc_refract.restype = Vec3
    L.orc_camera_new.argtypes = [Vec3, Vec3, Vec3, C.c_double, C.c_double, C.c_void_p]
    L.orc_raycaster_pixel_resolution.argtypes = [C.c_void_p, ImageParams]
    L.orc_raycaster_pixel_resolution.restype = C.c_double
    L.orc_raycaster_get_ray.argtypes = [C.c_void_p, ImageParams, C.c_double, C.c_double, C.c_void_p]
    L.orc_philox4x32_10.argtypes = [C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
    L.orc_philox_stream.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, d16]
    L.orc_surface_func.argtypes = [d16, Vec3]
    L.orc_surface_func.restype = C.c_double
    L.orc_surface_gradient.argtypes = [d16, Vec3]
    L.orc_surface_gradient.restype = Vec3
    L.orc_scene_create.argtypes = [C.c_void_p]
    L.orc_scene_create.restype = C.c_void_p
    L.orc_scene_destroy.argtypes = [C.c_void_p]
    L.orc_scene_build_bvh.argtypes = [C.c_void_p, C.c_uint64]
    L.orc_shape_bounding_box.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(Vec3), C.POINTER(Vec3)]
    L.orc_intersect_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_double, C.c_double, C.c_int, C.c_uint32,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p]
    L.orc_intersect_batch.restype = C.c_double
    L.orc_render.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32,
                             C.c_uint64, C.c_int, C.c_int, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]
    L.orc_render.restype = C.c_double
    L.orc_trace_pixel_samples.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint64, C.c_uint32,
                                          C.c_int, C.POINTER(Vec3)]
    L.orc_pixel_sample_colors.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32,
                                          C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint64, C.c_void_p]
    L.orc_pixels_sample_colors.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint64, C.c_void_p,
                                           C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint64, C.c_uint32, C.c_void_p]
    L.orc_groups_sample_colors.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64,
                                           C.c_uint32, C.c_uint64, C.c_uint32, C.c_void_p]
    L.orc_hardware_threads.restype = C.c_uint32
    L.orc_shape_hits.argtypes = [C.c_void_p, C.c_void_p, C.c_double, C.c_void_p]
    L.orc_solve_quartic.argtypes = [C.c_double] * 5 + [d16, d16]
    L.orc_perlin_noise.argtypes = [C.c_void_p, Vec3]
    L.orc_perlin_noise.restype = C.c_double
    L.orc_perlin_turb.argtypes = [C.c_void_p, Vec3, C.c_int]
    L.orc_perlin_turb.restype = C.c_double
    _lib = L
    return L


def hardware_threads() -> int:
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    return max(1, n)


def mat16(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float64).reshape(16)


def _p(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def mat_mul(a, b) -> np.ndarray:
    out = np.empty(16)
    lib().orc_mat_mul(_p(mat16(a)), _p(mat16(b)), _p(out))
    return out.reshape(4, 4)


def mat_rotate(deg) -> np.ndarray:
    out = np.empty(16)
    lib().orc_mat_rotate(Vec3(*deg), _p(out))
    return out.reshape(4, 4)


def transform_new(translate, rotate, scale):
    d, i = np.empty(16), np.empty(16)
    lib().orc_transform_new(Vec3(*translate), Vec3(*rotate), Vec3(*scale), _p(d), _p(i))
    return d.reshape(4, 4), i.reshape(4, 4)


def transform_point(m, p):
    return np.array(lib().orc_transform_point(_p(mat16(m)), Vec3(*p)).tuple())


def aabb_transform(mn, mx, m):
    a, b = Vec3(), Vec3()
    lib().orc_aabb_transform(Vec3(*mn), Vec3(*mx), _p(mat16(m)), C.byref(a), C.byref(b))
    return np.array(a.tuple()), np.array(b.tuple())


def camera_new(position, direction, up, focal_length, fov_rad) -> Camera:
    cam = Camera()
    lib().orc_camera_new(Vec3(*position), Vec3(*direction), Vec3(*up), focal_length, fov_rad, C.byref(cam))
    return cam


def pixel_resolution(cam: Camera, w: int, h: int) -> float:
    return lib().orc_raycaster_pixel_resolution(C.byref(cam), ImageParams(w, h))


def get_ray(cam: Camera, w: int, h: int, x: float, y: float) -> np.ndarray:
    r = Ray()
    lib().orc_raycaster_get_ray(C.byref(cam), ImageParams(w, h), x, y, C.byref(r))
    return np.array(r.origin.tuple() + r.direction.tuple())


def philox(ctr, key) -> np.ndarray:
    c = (C.c_uint32 * 4)(*ctr)
    k = (C.c_uint32 * 2)(*key)
    o = (C.c_uint32 * 4)()
    lib().orc_philox4x32_10(c, k, o)
    return np.array(list(o), dtype=np.uint32)


def philox_stream(seed, pixel, sample, event, n) -> np.ndarray:
    out = np.empty(n)
    lib().orc_philox_stream(seed, pixel, sample, event, n, _p(out))
    return out


def solve_quartic(a, b, c, d, e) -> np.ndarray:
    """solve_quantic_equation (src/algebra/equation.rs:17-67): the four complex roots"""
    re, im = np.empty(4), np.empty(4)
    lib().orc_solve_quartic(a, b, c, d, e, _p(re), _p(im))
    return re + 1j * im


def perlin_noise(table, p) -> float:
    """Perlin::noise (src/algebra/noise.rs:43-73) on an rt_perlin table (ctypes struct)"""
    return lib().orc_perlin_noise(C.addressof(table), Vec3(*map(float, p)))


def perlin_turb(table, p, depth=7) -> float:
    return lib().orc_perlin_turb(C.addressof(table), Vec3(*map(float, p)), depth)


def save_flat_scene(path: str, desc, cam, note: str = "") -> None:
    """Write an rt_scene_desc + camera as an .npz (tools/make_oracle_scenes.py): what the reference arm of bench.py
    loads instead of importing the product's scene loader."""
    n = desc.n_shapes
    arr = lambda ptr, shape, dt: np.ctypeslib.as_array(ptr, shape=shape).astype(dt).copy() if shape[0] else np.zeros(shape, dt)
    mats = np.array([(desc.materials[i].kind, desc.materials[i].texture, desc.materials[i].scalar)
                     for i in range(desc.n_materials)], dtype=np.float64).reshape(-1, 3)
    texs = np.array([(t.kind, t.odd, t.even, t.image, t.color.x, t.color.y, t.color.z)
                     for t in (desc.textures[i] for i in range(desc.n_textures))], dtype=np.float64).reshape(-1, 7)
    out = {"kind": arr(desc.kind, (n,), np.uint8), "flags": arr(desc.flags, (n,), np.uint8),
           "inverse": arr(desc.inverse, (n, 12), np.float64), "direct": arr(desc.direct, (n, 12), np.float64),
           "params": arr(desc.params, (n, 8), np.float64), "material": arr(desc.material, (n,), np.uint32),
           "materials": mats, "textures": texs, "note": np.array(note),
           "camera": np.array(cam.position.tuple() + cam.direction.tuple() + cam.up.tuple() + cam.right.tuple()
                              + (cam.fov_rad, cam.focal_length))}
    for i in range(desc.n_images):
        im = desc.images[i]
        out[f"image{i}"] = np.ctypeslib.as_array(im.rgba, shape=(im.height, im.width, 4)).copy()
    if desc.n_noise:
        out["noise"] = np.frombuffer(C.string_at(desc.noise, C.sizeof(Perlin) * desc.n_noise), dtype=np.uint8).copy()
    np.savez_compressed(path, **out)


def load_flat_scene(path: str):
    """-> (OracleScene, Camera) from a file written by save_flat_scene"""
    z = np.load(path)
    keep = {k: np.ascontiguousarray(z[k]) for k in z.files}
    d = SceneDesc()
    n = keep["kind"].shape[0]
    d.n_shapes = n
    ptr = lambda a, t: a.ctypes.data_as(C.POINTER(t))
    d.kind, d.flags = ptr(keep["kind"], C.c_uint8), ptr(keep["flags"], C.c_uint8)
    d.inverse, d.direct, d.params = (ptr(keep[k], C.c_double) for k in ("inverse", "direct", "params"))
    d.material = ptr(keep["material"], C.c_uint32)
    mats = (Material * max(len(keep["materials"]), 1))()
    for i, (k, t, s) in enumerate(keep["materials"]):
        mats[i].kind, mats[i].texture, mats[i].scalar = int(k), int(t), float(s)
    texs = (Texture * max(len(keep["textures"]), 1))()
    for i, row in enumerate(keep["textures"]):
        texs[i].kind, texs[i].odd, texs[i].even, texs[i].image = (int(v) for v in row[:4])
        texs[i].color = Vec3(*row[4:7])
    d.n_materials, d.materials = len(keep["materials"]), mats
    d.n_textures, d.textures = len(keep["textures"]), texs
    n_img = sum(1 for k in keep if k.startswith("image"))
    imgs = (Image * max(n_img, 1))()
    for i in range(n_img):
        a = keep[f"image{i}"]
        imgs[i].height, imgs[i].width, imgs[i].rgba = a.shape[0], a.shape[1], ptr(a, C.c_uint8)
    d.n_images, d.images = n_img, imgs
    if "noise" in keep:
        d.n_noise = keep["noise"].size // C.sizeof(Perlin)
        d.noise = C.cast(keep["noise"].ctypes.data, C.POINTER(Perlin))
    c = keep["camera"]
    cam = Camera()
    cam.position, cam.direction, cam.up, cam.right = (Vec3(*c[3 * i: 3 * i + 3]) for i in range(4))
    cam.fov_rad, cam.focal_length = float(c[12]), float(c[13])
    return OracleScene(d, keepalive=(keep, mats, texs, imgs)), cam


class OracleScene:
    """The oracle's decoded copy of a flat scene description (an rt_scene_desc)."""

    def __init__(self, desc: SceneDesc, keepalive=None):
        self._keep = keepalive
        self._h = lib().orc_scene_create(C.byref(desc))
        if not self._h:
            raise ValueError("oracle: invalid scene description")
        self._has_bvh = False

    def __del__(self):
        if getattr(self, "_h", None):
            lib().orc_scene_destroy(self._h)
            self._h = None

    def build_bvh(self, seed: int = 1):
        lib().orc_scene_build_bvh(self._h, seed)
        self._has_bvh = True

    def bounding_box(self, i: int):
        a, b = Vec3(), Vec3()
        lib().orc_shape_bounding_box(self._h, i, C.byref(a), C.byref(b))
        return np.array(a.tuple()), np.array(b.tuple())

    def intersect_batch(self, rays: np.ndarray, min_t=0.001, max_t=math.inf, use_bvh=False, threads=None,
                        counters=False):
        rays = np.ascontiguousarray(rays, dtype=np.float64).reshape(-1, 6)
        n = rays.shape[0]
        if use_bvh and not self._has_bvh:
            self.build_bvh()
        out = {"index": np.empty(n, np.int32), "t": np.empty(n), "normal": np.empty((n, 3)),
               "point": np.empty((n, 3)), "uv": np.empty((n, 2)), "front": np.empty(n, np.uint8)}
        cnt = np.zeros(5, np.uint64)
        vp = lambda a: a.ctypes.data_as(C.c_void_p)
        secs = lib().orc_intersect_batch(self._h, vp(rays), n, min_t, max_t, int(use_bvh), threads or hardware_threads(),
                                         vp(out["index"]), vp(out["t"]), vp(out["normal"]), vp(out["point"]),
                                         vp(out["uv"]), vp(out["front"]), vp(cnt) if counters else None)
        out["seconds"] = secs
        if counters:
            out["counters"] = dict(zip(["segments", "shape_tests", "march_steps", "march_rays", "aabb_tests"],
                                       [int(x) for x in cnt]))
        return out

    def render(self, cam: Camera, width, height, spp, depth, seed=0, rng="philox", use_bvh=False, threads=None,
               stride=(1, 1), counters=False):
        buf = np.zeros((height, width, 3))
        cnt = np.zeros(5, np.uint64)
        if use_bvh and not self._has_bvh:
            self.build_bvh()
        secs = lib().orc_render(self._h, C.byref(cam), width, height, spp, depth, seed, 0 if rng == "philox" else 1,
                                int(use_bvh), threads or hardware_threads(), stride[0], stride[1],
                                buf.ctypes.data_as(C.c_void_p), cnt.ctypes.data_as(C.c_void_p) if counters else None)
        info = {"seconds": secs}
        if counters:
            info["counters"] = dict(zip(["segments", "shape_tests", "march_steps", "march_rays", "aabb_tests"],
                                        [int(x) for x in cnt]))
        return buf, info

    def shape_hits(self, ray, n_shapes: int, min_t=0.001) -> np.ndarray:
        """Shape::ray_hit of EVERY shape for one ray with max_t = +inf (a marched shape: its bound); uint8[n_shapes]"""
        ray = np.ascontiguousarray(ray, dtype=np.float64).reshape(6)
        out = np.zeros(n_shapes, np.uint8)
        lib().orc_shape_hits(self._h, ray.ctypes.data_as(C.c_void_p), min_t, out.ctypes.data_as(C.c_void_p))
        return out

    def trace_pixel_samples(self, rays: np.ndarray, depth, seed=0, pixel_index=0, use_bvh=False):
        rays = np.ascontiguousarray(rays, dtype=np.float64).reshape(-1, 6)
        mean = Vec3()
        lib().orc_trace_pixel_samples(self._h, rays.ctypes.data_as(C.c_void_p), rays.shape[0], depth, seed, pixel_index,
                                      int(use_bvh), C.byref(mean))
        return np.array(mean.tuple())

    def group_sample_colors(self, rays: np.ndarray, offsets, pixel_index, depth, seed=0, threads=None):
        """Per-ray FP64 radiance of caller rays in groups (trace_pixel_samples_group): ray r of group g, rays
        offsets[g] .. offsets[g+1]-1, is sample r - offsets[g] of pixel pixel_index[g].  float64[n_rays, 3]."""
        rays = np.ascontiguousarray(rays, dtype=np.float64).reshape(-1, 6)
        off = np.ascontiguousarray(offsets, dtype=np.uint64).reshape(-1)
        pix = np.ascontiguousarray(pixel_index, dtype=np.uint32).reshape(-1)
        if off.size != pix.size + 1 or off[0] != 0 or int(off[-1]) != rays.shape[0] or (np.diff(off.astype(np.int64)) < 0).any():
            raise ValueError("offsets must rise from 0 to len(rays), one more than pixel_index")
        out = np.empty((rays.shape[0], 3))
        vp = lambda a: a.ctypes.data_as(C.c_void_p)
        lib().orc_groups_sample_colors(self._h, vp(rays), rays.shape[0], vp(off), vp(pix), pix.size, depth, seed,
                                       threads or hardware_threads(), vp(out))
        return out

    def pixel_sample_colors(self, cam: Camera, width, height, x, y, spp, depth, seed=0):
        out = np.empty((spp, 3))
        lib().orc_pixel_sample_colors(self._h, C.byref(cam), width, height, x, y, spp, depth, seed,
                                      out.ctypes.data_as(C.c_void_p))
        return out

    def frame_sample_colors(self, cam: Camera, width, height, spp, depth, seed=0, pixels=None, sample_base=0,
                            threads=None):
        """Per-sample FP64 radiance (Philox schedule) of samples sample_base .. sample_base + spp - 1 of the pixels
        `pixels` (indices x + y*width; None = every pixel): float64[len(pixels), spp, 3]."""
        if pixels is None:
            pixels = np.arange(width * height)
        pix = np.ascontiguousarray(pixels, dtype=np.uint32).reshape(-1)
        out = np.empty((pix.size, spp, 3))
        lib().orc_pixels_sample_colors(self._h, C.byref(cam), width, height, pix.size, pix.ctypes.data_as(C.c_void_p),
                                       sample_base, spp, depth, seed, threads or hardware_threads(),
                                       out.ctypes.data_as(C.c_void_p))
        return out
