"""ctypes bindings of include/rt_b200.h (the C-ABI drop-in boundary) and include/rt_b200_host.h
(the C shim over the C++ host mirror).  Loading fails loudly when the libraries are not built:
there is no Python or CPU fallback for any compute entry point."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
CORE_SO = os.path.join(HERE, "librt_b200.so")
HOST_SO = os.path.join(HERE, "librt_b200_host.so")

RT_OK = 0
RT_ERR_INVALID, RT_ERR_NO_DEVICE, RT_ERR_CUDA, RT_ERR_STATE, RT_ERR_NOMEM = -1, -2, -3, -4, -5
RT_ISECT_BRUTE, RT_ISECT_FAST, RT_ISECT_VERIFY = 0, 1, 2
RT_BOUNCE_MISS, RT_BOUNCE_SCATTER, RT_BOUNCE_EMIT = 0, 1, 2
RT_SHAPE_SPHERE, RT_SHAPE_CUBE, RT_SHAPE_RECTANGLE, RT_SHAPE_MARCH, RT_SHAPE_TORUS = 0, 1, 2, 3, 4
RT_SURF_HEART, RT_SURF_SINE, RT_SURF_STAR, RT_SURF_DUPIN, RT_SURF_HUNTS, RT_SURF_CUSHION = range(6)
RT_MAT_LAMBERTIAN, RT_MAT_METAL, RT_MAT_DIELECTRIC, RT_MAT_DIFFUSE_LIGHT, RT_MAT_EMPTY = range(5)
RT_TEX_SOLID, RT_TEX_CHECKER, RT_TEX_UV_CHECKER, RT_TEX_IMAGE, RT_TEX_NOISE = range(5)
RT_SHAPE_PARAMS = 8


class Vec3(C.Structure):
    _fields_ = [("x", C.c_double), ("y", C.c_double), ("z", C.c_double)]

    def __init__(self, x=0.0, y=0.0, z=0.0):
        super().__init__(float(x), float(y), float(z))

    def tuple(self):
        return (self.x, self.y, self.z)


class Ray(C.Structure):
    _fields_ = [("origin", Vec3), ("direction", Vec3)]


class Camera(C.Structure):
    _fields_ = [("position", Vec3), ("direction", Vec3), ("up", Vec3), ("right", Vec3),
                ("fov_rad", C.c_double), ("focal_length", C.c_double)]


class ImageParams(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32)]


class Material(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("texture", C.c_uint32), ("scalar", C.c_double)]


class Texture(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("odd", C.c_uint32), ("even", C.c_uint32), ("image", C.c_uint32),
                ("color", Vec3)]


class Image(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("rgba", C.POINTER(C.c_uint8))]


class Perlin(C.Structure):
    _fields_ = [("perm_x", C.c_uint32 * 256), ("perm_y", C.c_uint32 * 256), ("perm_z", C.c_uint32 * 256),
                ("ranvec", Vec3 * 256)]


class SceneDesc(C.Structure):
    _fields_ = [
        ("n_shapes", C.c_uint32),
        ("kind", C.POINTER(C.c_uint8)),
        ("flags", C.POINTER(C.c_uint8)),
        ("inverse", C.POINTER(C.c_double)),
        ("direct", C.POINTER(C.c_double)),
        ("params", C.POINTER(C.c_double)),
        ("material", C.POINTER(C.c_uint32)),
        ("n_materials", C.c_uint32),
        ("materials", C.POINTER(Material)),
        ("n_textures", C.c_uint32),
        ("textures", C.POINTER(Texture)),
        ("n_images", C.c_uint32),
        ("images", C.POINTER(Image)),
        ("n_noise", C.c_uint32),
        ("noise", C.POINTER(Perlin)),
    ]


class RenderParams(C.Structure):
    _fields_ = [
        ("image", ImageParams),
        ("samples_number", C.c_uint32),
        ("max_depth", C.c_uint32),
        ("seed", C.c_uint64),
        ("shard_count", C.c_uint32),
        ("shard_index", C.c_uint32),
        ("tile_width", C.c_uint32),
        ("tile_height", C.c_uint32),
    ]


class AdaptiveParams(C.Structure):
    _fields_ = [
        ("min_samples", C.c_uint32),
        ("rel_error", C.c_double),
        ("abs_error", C.c_double),
    ]


class FeaturePlanes(C.Structure):   # rt_feature_planes: w * h values each, NULL = not wanted
    _fields_ = [("albedo", C.c_void_p), ("normal", C.c_void_p), ("depth", C.c_void_p), ("coverage", C.c_void_p),
                ("shape", C.c_void_p)]



class Stats(C.Structure):
    _fields_ = [
        ("kernel_launches", C.c_uint64),
        ("paths", C.c_uint64),
        ("segments", C.c_uint64),
        ("shape_tests", C.c_uint64),
        ("cull_tests", C.c_uint64),
        ("march_steps", C.c_uint64),
        ("march_rays", C.c_uint64),
        ("march_long_rays", C.c_uint64),
        ("march_max_evals", C.c_uint64),
        ("last_frame_ms", C.c_double),
        ("last_intersect_ms", C.c_double),
        ("verify_rays", C.c_uint64),
        ("verify_false_culls", C.c_uint64),
        ("ms_raygen", C.c_double),
        ("ms_extend", C.c_double),
        ("ms_march", C.c_double),
        ("ms_shade", C.c_double),
        ("ms_resolve", C.c_double),
        ("launches_extend", C.c_uint64),
        ("launches_march", C.c_uint64),
        ("launches_shade", C.c_uint64),
        ("march_prof", C.c_uint64 * 8),
    ]


# every symbol include/rt_b200.h declares: name -> (restype, argtypes)
CORE_SYMBOLS = {
    "rt_abi_version": (C.c_int, []),
    "rt_last_error": (C.c_char_p, []),
    "rt_device_count": (C.c_int, []),
    "rt_scene_create": (C.c_int, [C.POINTER(SceneDesc), C.c_int, C.POINTER(C.c_void_p)]),
    "rt_scene_destroy": (None, [C.c_void_p]),
    "rt_scene_create_multi": (C.c_int, [C.POINTER(SceneDesc), C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_void_p)]),
    "rt_scene_device_count": (C.c_int, [C.c_void_p]),
    "rt_scene_update": (C.c_int, [C.c_void_p, C.POINTER(SceneDesc)]),
    "rt_scene_update_transforms": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rt_intersect_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_double, C.c_double, C.c_int,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rt_intersect_batch_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_double, C.c_double, C.c_int,
                                            C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_void_p]),
    "rt_occluded_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_double, C.c_double, C.c_void_p, C.c_int,
                                    C.c_void_p]),
    "rt_occluded_batch_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_double, C.c_double, C.c_void_p,
                                           C.c_int, C.c_void_p, C.c_void_p]),
    "rt_scatter_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint64, C.c_double,
                                   C.c_double, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rt_scatter_batch_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint64,
                                          C.c_double, C.c_double, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p, C.c_void_p]),
    "rt_render_start": (C.c_int, [C.c_void_p, C.POINTER(Camera), C.POINTER(RenderParams)]),
    "rt_render_poll": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_int)]),
    "rt_render_wait": (C.c_int, [C.c_void_p, C.c_void_p]),
    "rt_render_stop": (C.c_int, [C.c_void_p]),
    "rt_render_set_accumulate": (C.c_int, [C.c_void_p, C.c_int]),
    "rt_render_accumulated_samples": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint32)]),
    "rt_render_start_adaptive": (C.c_int, [C.c_void_p, C.POINTER(Camera), C.POINTER(RenderParams),
                                           C.POINTER(AdaptiveParams)]),
    "rt_render_pixel_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "rt_render_start_counts": (C.c_int, [C.c_void_p, C.POINTER(Camera), C.POINTER(RenderParams), C.c_void_p]),
    "rt_render_start_views": (C.c_int, [C.c_void_p, C.POINTER(Camera), C.c_uint32, C.POINTER(RenderParams)]),
    "rt_render_start_layers": (C.c_int, [C.c_void_p, C.POINTER(Camera), C.POINTER(RenderParams), C.c_uint32]),
    "rt_render_layers": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]),
    "rt_render_device_layers": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]),
    "rt_assemble_layers": (C.c_int, [C.c_void_p, C.POINTER(RenderParams), C.c_uint32, C.POINTER(C.c_void_p),
                                     C.POINTER(C.c_void_p), C.c_void_p, C.c_void_p]),
    "rt_render_start_features": (C.c_int, [C.c_void_p, C.POINTER(Camera), C.POINTER(RenderParams)]),
    "rt_render_features": (C.c_int, [C.c_void_p, C.POINTER(FeaturePlanes), C.POINTER(FeaturePlanes)]),
    "rt_render_device_features": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]),
    "rt_assemble_features": (C.c_int, [C.c_void_p, C.POINTER(RenderParams), C.POINTER(C.c_void_p),
                                       C.POINTER(FeaturePlanes), C.c_void_p]),
    "rt_render_device_result": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]),
    "rt_shard_float4_count": (C.c_uint64, [C.POINTER(RenderParams), C.c_uint32]),
    "rt_assemble_frame": (C.c_int, [C.c_void_p, C.POINTER(RenderParams), C.POINTER(C.c_void_p), C.c_void_p,
                                    C.c_void_p]),
    "rt_render_device_frame": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]),
    "rt_tonemap_rgba8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "rt_tonemap_rgba8_device": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.c_void_p, C.POINTER(C.c_uint64)]),
    "rt_trace_pixel_samples": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint64, C.c_uint32,
                                         C.POINTER(Vec3)]),
    "rt_trace_pixel_samples_group": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint32,
                                               C.c_uint32, C.c_uint64, C.c_void_p]),
    "rt_trace_pixel_samples_group_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p,
                                                      C.c_uint32, C.c_uint32, C.c_uint64, C.c_void_p, C.c_void_p]),
    "rt_get_stats": (C.c_int, [C.c_void_p, C.POINTER(Stats)]),
    "rt_reset_stats": (C.c_int, [C.c_void_p]),
    "rt_set_counters": (C.c_int, [C.c_void_p, C.c_int]),
    "rt_set_kernel_timing": (C.c_int, [C.c_void_p, C.c_int]),
    "rt_march_region_bounds": (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "rt_advance_exact": (C.c_int, [C.c_double, C.c_double, C.c_int64, C.POINTER(C.c_double)]),
    "rt_div3_exact": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "rt_march_candidates_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_double, C.c_double, C.c_double,
                                          C.c_int, C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64)]),
    "rt_bernstein_clear": (C.c_int, [C.c_void_p, C.c_int, C.c_double, C.c_double, C.POINTER(C.c_int)]),
    "rt_cull_reached": (C.c_int, [C.POINTER(SceneDesc), C.c_void_p, C.c_uint64, C.c_void_p]),
    "rt_cull_tree_check": (C.c_int, [C.POINTER(SceneDesc), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32),
                                    C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_double)]),
    "rt_cull_refit_check": (C.c_int, [C.POINTER(SceneDesc), C.c_uint32, C.c_void_p, C.c_void_p, C.POINTER(C.c_double)]),
    "rt_measure_peaks": (C.c_int, [C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
}

IMAGE_LOADER = C.CFUNCTYPE(C.c_int, C.c_char_p, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32),
                           C.POINTER(C.POINTER(C.c_uint8)))

HOST_SYMBOLS = {
    "rth_last_error": (C.c_char_p, []),
    "rth_set_image_loader": (None, [IMAGE_LOADER]),
    "rth_scene_from_json": (C.c_int, [C.c_char_p, C.c_uint64, C.c_int, C.POINTER(C.c_void_p)]),
    "rth_scene_free": (None, [C.c_void_p]),
    "rth_scene_desc": (C.c_int, [C.c_void_p, C.POINTER(SceneDesc)]),
    "rth_scene_camera": (C.c_int, [C.c_void_p, C.POINTER(Camera)]),
    "rth_scene_shape_count": (C.c_uint32, [C.c_void_p]),
    "rth_scene_shape_name": (C.c_char_p, [C.c_void_p, C.c_uint32]),
    "rth_scene_material_name": (C.c_char_p, [C.c_void_p, C.c_uint32]),
    "rth_scene_assign_material": (C.c_int, [C.c_void_p, C.c_uint32, C.c_char_p]),
    "rth_scene_set_transforms": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rth_scene_device": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]),
    "rth_scene_device_multi": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_void_p)]),
    "rth_camera_new": (C.c_int, [Vec3, Vec3, Vec3, C.c_double, C.c_double, C.POINTER(Camera)]),
    "rth_transform_new": (C.c_int, [Vec3, Vec3, Vec3, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "rth_renderer_new": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_int, C.c_uint64, C.POINTER(C.c_void_p)]),
    "rth_renderer_new_multi": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_int, C.POINTER(C.c_int), C.c_uint64,
                                         C.POINTER(C.c_void_p)]),
    "rth_renderer_free": (None, [C.c_void_p]),
    "rth_renderer_start_rendering": (C.c_int, [C.c_void_p, C.POINTER(Camera), ImageParams, C.c_uint32]),
    "rth_renderer_render_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_int)]),
    "rth_renderer_stop_rendering": (C.c_int, [C.c_void_p]),
    "rth_save_png": (C.c_int, [C.c_char_p, C.c_void_p, C.c_uint32, C.c_uint32]),
}


class NativeLibraryMissing(ImportError):
    pass


def _load(path: str, symbols: dict) -> C.CDLL:
    if not os.path.exists(path):
        raise NativeLibraryMissing(
            f"{path} is not built; run `python -m rs_pathtracing_b200.build` (needs nvcc). "
            "The path-tracing core has no Python/CPU fallback.")
    lib = C.CDLL(path, mode=C.RTLD_GLOBAL)
    for name, (restype, argtypes) in symbols.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = restype
        fn.argtypes = argtypes
    return lib


_core = None
_host = None


def core() -> C.CDLL:
    global _core
    if _core is None:
        _core = _load(CORE_SO, CORE_SYMBOLS)
    return _core


def host() -> C.CDLL:
    global _host
    if _host is None:
        core()  # librt_b200_host.so depends on it ($ORIGIN rpath)
        _host = _load(HOST_SO, HOST_SYMBOLS)
    return _host
