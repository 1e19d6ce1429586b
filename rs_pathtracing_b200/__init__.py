"""rs_pathtracing_b200 — B200-native path-tracing core for rs-pathtracing.

Only what the hot path needs: csrc/ (the sm_100a CUDA kernels behind the C ABI in include/rt_b200.h
and the C++ host mirror of the reference crate's interface), the ctypes bindings and a thin Python
face with the reference's names.  Importing this package requires the native libraries to be built
(`python -m rs_pathtracing_b200.build`); nothing here falls back to Python or CPU compute.
"""
from . import _ffi
from ._ffi import (Camera, ImageParams, Ray, RenderParams, Stats, Vec3, NativeLibraryMissing,
                   RT_ISECT_BRUTE, RT_ISECT_FAST, RT_ISECT_VERIFY, RT_BOUNCE_MISS, RT_BOUNCE_SCATTER, RT_BOUNCE_EMIT)
from .api import (GpuRenderer, RtError, Scene, camera_new, device_count, feature_means, group_means, layer_means,
                  make_rays, measure_peaks, path_levels, save_png, shadow_rays, tonemap_rgba8, trace_paths)

__all__ = [
    "Camera", "ImageParams", "Ray", "RenderParams", "Stats", "Vec3", "NativeLibraryMissing",
    "RT_ISECT_BRUTE", "RT_ISECT_FAST", "RT_ISECT_VERIFY", "RT_BOUNCE_MISS", "RT_BOUNCE_SCATTER", "RT_BOUNCE_EMIT",
    "GpuRenderer", "RtError", "Scene", "camera_new", "device_count", "feature_means", "group_means", "layer_means",
    "make_rays", "measure_peaks", "path_levels", "save_png", "shadow_rays", "tonemap_rgba8", "trace_paths",
]
