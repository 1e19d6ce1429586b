"""Python face of the host mirror: Scene / Camera / ImageParams / GpuRenderer with the reference's
method names (src/world/mod.rs, src/camera/mod.rs, src/renderer/mod.rs:47-56).  Every method is a
thin call into the native libraries; numpy only carries the buffers."""
from __future__ import annotations

import ctypes as C
import math
import os
from typing import Optional

import numpy as np

from . import _ffi
from ._ffi import Camera, ImageParams, RenderParams, Stats, Vec3


class RtError(RuntimeError):
    pass


def _check(rc: int, host: bool = False) -> None:
    if rc != _ffi.RT_OK:
        lib = _ffi.host() if host else _ffi.core()
        msg = (lib.rth_last_error() if host else lib.rt_last_error()) or b""
        if host and not msg:
            msg = _ffi.core().rt_last_error() or b""
        raise RtError(f"rt_b200 error {rc}: {msg.decode(errors='replace')}")


def device_count() -> int:
    return _ffi.core().rt_device_count()


def vec3(v) -> Vec3:
    return v if isinstance(v, Vec3) else Vec3(*v)


def camera_new(position, direction, up, focal_length: float, fov_rad: float) -> Camera:
    """Camera::new (src/camera/mod.rs:71-88); fov in radians."""
    cam = Camera()
    _check(_ffi.host().rth_camera_new(vec3(position), vec3(direction), vec3(up), focal_length, fov_rad,
                                      C.byref(cam)), host=True)
    return cam


_pil_loader_ref = None


def _install_pil_loader() -> None:
    """Register a PIL-based decoder for ImageTexture files that are not binary PPM
    (stands in for image::open, src/world/texture.rs:128-139)."""
    global _pil_loader_ref
    if _pil_loader_ref is not None:
        return
    libc = C.CDLL(None)
    libc.malloc.restype = C.c_void_p
    libc.malloc.argtypes = [C.c_size_t]

    def loader(filename, w, h, out):
        try:
            from PIL import Image as PILImage
            im = PILImage.open(filename.decode()).convert("RGBA")
            data = im.tobytes()
            buf = libc.malloc(len(data))
            C.memmove(buf, data, len(data))
            w[0], h[0] = im.width, im.height
            out[0] = C.cast(buf, C.POINTER(C.c_uint8))
            return 1
        except Exception:
            return 0

    _pil_loader_ref = _ffi.IMAGE_LOADER(loader)
    _ffi.host().rth_set_image_loader(_pil_loader_ref)


def make_rays(origins: np.ndarray, directions: np.ndarray, normalize: bool = True) -> np.ndarray:
    """(n,3),(n,3) -> (n,6) float64 array laid out like rt_ray.  normalize=True applies Ray::new
    (src/world/ray.rs:12-17) with the reference's arithmetic: d / sqrt((x*x + y*y) + z*z)."""
    o = np.ascontiguousarray(origins, dtype=np.float64).reshape(-1, 3)
    d = np.ascontiguousarray(directions, dtype=np.float64).reshape(-1, 3)
    if normalize:
        ln = np.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1] + d[:, 2] * d[:, 2])
        d = d / ln[:, None]
    return np.ascontiguousarray(np.concatenate([o, d], axis=1))


class Scene:
    """world::Scene (src/world/mod.rs:20-49)."""

    def __init__(self, handle):
        self._h = handle
        self._keep = None
        self._device = 0   # the device the helpers below address by default: the last one asked for explicitly

    @classmethod
    def from_json(cls, data: str, random_spheres_seed: int = 1, add_random_spheres: bool = True,
                  base_dir: Optional[str] = None) -> "Scene":
        """Scene::from_json.  `data` is the JSON text.  ImageTexture paths are cwd-relative like the
        reference's; pass base_dir to resolve them against another directory."""
        _install_pil_loader()
        h = C.c_void_p()
        cwd = os.getcwd()
        try:
            if base_dir:
                os.chdir(base_dir)
            rc = _ffi.host().rth_scene_from_json(data.encode(), random_spheres_seed, int(add_random_spheres),
                                                 C.byref(h))
        finally:
            os.chdir(cwd)
        _check(rc, host=True)
        return cls(h)

    @classmethod
    def from_file(cls, path: str, random_spheres_seed: int = 1, add_random_spheres: bool = True) -> "Scene":
        with open(path) as f:
            text = f.read()
        # texture paths in the scene files are written relative to the repository root
        root = os.path.dirname(os.path.dirname(os.path.abspath(path)))
        return cls.from_json(text, random_spheres_seed, add_random_spheres, base_dir=root)

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            try:
                _ffi.host().rth_scene_free(h)
            except Exception:
                pass

    def camera(self) -> Camera:
        cam = Camera()
        _check(_ffi.host().rth_scene_camera(self._h, C.byref(cam)), host=True)
        return cam

    def desc(self) -> _ffi.SceneDesc:
        d = _ffi.SceneDesc()
        _check(_ffi.host().rth_scene_desc(self._h, C.byref(d)), host=True)
        d._owner = self  # the arrays live inside the native scene: keep it alive with the view
        return d

    @property
    def shape_count(self) -> int:
        return _ffi.host().rth_scene_shape_count(self._h)

    def shape_name(self, i: int) -> str:
        return _ffi.host().rth_scene_shape_name(self._h, i).decode()

    def shape_kinds(self) -> np.ndarray:
        d = self.desc()
        return np.ctypeslib.as_array(d.kind, shape=(d.n_shapes,)).copy()

    def assign_material(self, shape_index: int, material_name: str) -> None:
        _check(_ffi.host().rth_scene_assign_material(self._h, shape_index, material_name.encode()), host=True)

    def device_scene(self, device: Optional[int] = None) -> C.c_void_p:
        """the rt_scene handle on `device` (one per device, created on first use, alive as long as this Scene).
        device=None: the device last asked for explicitly (a renderer's), 0 at first."""
        if device is None:
            device = self._device
        else:
            self._device = device
        out = C.c_void_p()
        _check(_ffi.host().rth_scene_device(self._h, device, C.byref(out)), host=True)
        return out

    def device_scene_multi(self, devices) -> C.c_void_p:
        """ONE rt_scene handle over several devices (rt_scene_create_multi): whole-frame renders are sharded over them"""
        ids = (C.c_int * len(devices))(*devices)
        out = C.c_void_p()
        _check(_ffi.host().rth_scene_device_multi(self._h, len(devices), ids, C.byref(out)), host=True)
        return out

    # Scene::closest_hit (src/world/mod.rs:42-44) on a batch
    def closest_hit(self, rays: np.ndarray, min_t: float = 0.001, max_t: float = math.inf,
                    mode: int = _ffi.RT_ISECT_BRUTE, device: Optional[int] = None, want=("index", "t", "normal", "point", "uv", "front")):
        rays = np.ascontiguousarray(rays, dtype=np.float64).reshape(-1, 6)
        n = rays.shape[0]
        out = {
            "index": np.empty(n, np.int32) if "index" in want else None,
            "t": np.empty(n, np.float64) if "t" in want else None,
            "normal": np.empty((n, 3), np.float64) if "normal" in want else None,
            "point": np.empty((n, 3), np.float64) if "point" in want else None,
            "uv": np.empty((n, 2), np.float64) if "uv" in want else None,
            "front": np.empty(n, np.uint8) if "front" in want else None,
        }
        p = lambda a: a.ctypes.data_as(C.c_void_p) if a is not None else None
        _check(_ffi.core().rt_intersect_batch(self.device_scene(device), p(rays), n, min_t, max_t, mode, p(out["index"]),
                                              p(out["t"]), p(out["normal"]), p(out["point"]), p(out["uv"]),
                                              p(out["front"])))
        return {k: v for k, v in out.items() if v is not None}

    def trace_pixel_samples(self, rays: np.ndarray, depth: int, seed: int = 0, pixel_index: int = 0,
                            device: Optional[int] = None):
        """renderer::trace_pixel_samples (src/renderer/mod.rs:151-155)."""
        rays = np.ascontiguousarray(rays, dtype=np.float64).reshape(-1, 6)
        mean = Vec3()
        _check(_ffi.core().rt_trace_pixel_samples(self.device_scene(device), rays.ctypes.data_as(C.c_void_p),
                                                  rays.shape[0], depth, seed, pixel_index, C.byref(mean)))
        return np.array(mean.tuple())

    def trace_pixel_samples_group(self, rays, offsets, pixel_index, depth: int, seed: int = 0,
                                  device: Optional[int] = None):
        """renderer::trace_pixel_samples_group (src/renderer/mod.rs:127-149): group g = rays[offsets[g]:offsets[g+1]],
        the samples of pixel pixel_index[g]; returns the (g, 3) per-group means (NaN for an empty group).
        rays: numpy (n, 6) float64 -> numpy result after the host round trip; or a contiguous float64 CUDA torch tensor
        (n, 6) on the scene's device -> a torch tensor on that device, queued on torch's current stream without a host
        synchronisation.  offsets / pixel_index are host arrays in both cases."""
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64).reshape(-1)
        pixel_index = np.ascontiguousarray(pixel_index, dtype=np.uint32).reshape(-1)
        n_groups = pixel_index.shape[0]
        if offsets.shape[0] != n_groups + 1:
            raise ValueError(f"offsets needs n_groups + 1 = {n_groups + 1} entries, got {offsets.shape[0]}")
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        if type(rays).__module__.split(".")[0] == "torch":
            import torch
            if not (rays.is_cuda and rays.dtype == torch.float64 and rays.dim() == 2 and rays.shape[1] == 6
                    and rays.is_contiguous()):
                raise ValueError("rays: a contiguous float64 CUDA tensor of shape (n, 6)")
            h = self.device_scene(device)
            if rays.device.index != self._device:
                raise ValueError(f"rays are on {rays.device}, the scene's device is cuda:{self._device}")
            means = torch.empty((n_groups, 3), dtype=torch.float64, device=rays.device)
            # torch's default stream is the legacy default stream (handle 0), which the ABI names cudaStreamLegacy = 0x1
            stream = torch.cuda.current_stream(rays.device).cuda_stream or 1
            _check(_ffi.core().rt_trace_pixel_samples_group_device(h, rays.data_ptr(), rays.shape[0], p(offsets),
                                                                   p(pixel_index), n_groups, depth, seed,
                                                                   means.data_ptr(), stream))
            return means
        rays = np.ascontiguousarray(rays, dtype=np.float64).reshape(-1, 6)
        means = np.empty((n_groups, 3), np.float64)
        _check(_ffi.core().rt_trace_pixel_samples_group(self.device_scene(device), p(rays), rays.shape[0], p(offsets),
                                                        p(pixel_index), n_groups, depth, seed, p(means)))
        return means

    def stats(self, device: Optional[int] = None) -> Stats:
        s = Stats()
        _check(_ffi.core().rt_get_stats(self.device_scene(device), C.byref(s)))
        return s

    def reset_stats(self, device: Optional[int] = None) -> None:
        _check(_ffi.core().rt_reset_stats(self.device_scene(device)))

    def set_counters(self, enabled: bool, device: Optional[int] = None) -> None:
        _check(_ffi.core().rt_set_counters(self.device_scene(device), int(enabled)))

    def set_kernel_timing(self, enabled: bool, device: Optional[int] = None) -> None:
        _check(_ffi.core().rt_set_kernel_timing(self.device_scene(device), int(enabled)))


class GpuRenderer:
    """Drop-in for step_by_step::ThreadPoolRenderer (src/renderer/step_by_step.rs:37) implementing the
    Renderer trait (src/renderer/mod.rs:47-56)."""

    def __init__(self, scene: Scene, thread_number: int = 0, depth: int = 50, device: int = 0, seed: int = 0,
                 devices=None):
        """devices: a list of device indices -> ONE renderer (one process, one handle) that shards every frame
        over all of them by interleaved tiles; the frame is the single-device one, bit for bit"""
        self.scene = scene
        self.depth = depth
        self.seed = seed
        self.devices = list(devices) if devices else None
        self.device = self.devices[0] if self.devices else device
        scene._device = self.device
        self._h = C.c_void_p()
        if self.devices and len(self.devices) > 1:
            ids = (C.c_int * len(self.devices))(*self.devices)
            _check(_ffi.host().rth_renderer_new_multi(scene._h, thread_number, depth, len(self.devices), ids, seed,
                                                      C.byref(self._h)), host=True)
        else:
            _check(_ffi.host().rth_renderer_new(scene._h, thread_number, depth, self.device, seed, C.byref(self._h)),
                   host=True)

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            try:
                _ffi.host().rth_renderer_free(h)
            except Exception:
                pass

    def start_rendering(self, camera: Camera, img_params: ImageParams, samples_number: int) -> None:
        _check(_ffi.host().rth_renderer_start_rendering(self._h, C.byref(camera), img_params, samples_number), host=True)

    def render_step(self, buffer: np.ndarray) -> bool:
        """buffer: float64 array of shape (h*w, 3) or (h, w, 3), index x + y*w; returns True when complete."""
        assert buffer.dtype == np.float64 and buffer.flags["C_CONTIGUOUS"]
        done = C.c_int(0)
        _check(_ffi.host().rth_renderer_render_step(self._h, buffer.ctypes.data_as(C.c_void_p), buffer.size // 3,
                                                    C.byref(done)), host=True)
        return bool(done.value)

    def stop_rendering(self) -> None:
        _check(_ffi.host().rth_renderer_stop_rendering(self._h), host=True)

    def render(self, camera: Camera, width: int, height: int, samples_number: int) -> np.ndarray:
        """start_rendering + poll render_step until it returns True (what the bins' loop does)."""
        buf = np.zeros((height, width, 3), np.float64)
        self.start_rendering(camera, ImageParams(width, height), samples_number)
        while not self.render_step(buf):
            pass
        return buf

    def render_adaptive(self, camera: Camera, width: int, height: int, samples_number: int, min_samples: int,
                        rel_error: float, abs_error: float = 0.0):
        """An adaptive frame (rt_render_start_adaptive) on this renderer's device, depth and seed: returns
        (frame[h, w, 3] float64, counts[h, w] uint32 samples per pixel, std_error[h, w] of each pixel's mean
        luminance).  Single-device renderers only."""
        if self.devices and len(self.devices) > 1:
            raise ValueError("adaptive sampling renders on one device")
        h = self.scene.device_scene(self.device)
        params = render_params(width, height, samples_number, self.depth, self.seed)
        render_start_adaptive(h, camera, params, min_samples, rel_error, abs_error)
        frame = np.zeros((height, width, 3), np.float64)
        render_wait(h, frame)
        counts, moments = render_pixel_stats(h)
        return frame, counts, standard_error(counts, moments)


def tonemap_rgba8(scene: Scene, frame: np.ndarray, device: Optional[int] = None) -> np.ndarray:
    """src/bin/main_raylib.rs:239-247 on the device."""
    frame = np.ascontiguousarray(frame, dtype=np.float64)
    n = frame.size // 3
    out = np.empty((n, 4), np.uint8)
    _check(_ffi.core().rt_tonemap_rgba8(scene.device_scene(device), frame.ctypes.data_as(C.c_void_p), n,
                                        out.ctypes.data_as(C.c_void_p)))
    return out.reshape(frame.shape[:-1] + (4,))


def tonemap_last_frame(dev_scene, n_pixels_hint: int = 0) -> np.ndarray:
    """rt_tonemap_rgba8_device: the frame the library holds on the device -> (n, 4) uint8 on the host; only the 4
    bytes per pixel cross the bus"""
    n = C.c_uint64(0)
    ptr = C.c_void_p()
    frame_ptr = C.c_void_p()
    _check(_ffi.core().rt_render_device_frame(dev_scene, C.byref(frame_ptr), C.byref(n)))
    out = np.empty((n.value, 4), np.uint8)
    _check(_ffi.core().rt_tonemap_rgba8_device(dev_scene, C.byref(ptr), out.ctypes.data_as(C.c_void_p), C.byref(n)))
    return out


def save_png(path: str, rgba: np.ndarray) -> None:
    """image::save_buffer of the bins (main_raylib.rs:64-75): (h, w, 4) uint8 -> PNG"""
    rgba = np.ascontiguousarray(rgba, dtype=np.uint8)
    if rgba.ndim != 3 or rgba.shape[2] != 4:
        raise ValueError("rgba must have shape (h, w, 4)")
    _check(_ffi.host().rth_save_png(path.encode(), rgba.ctypes.data_as(C.c_void_p), rgba.shape[1], rgba.shape[0]),
           host=True)


def measure_peaks(device: int = 0):
    a, b = C.c_double(), C.c_double()
    _check(_ffi.core().rt_measure_peaks(device, C.byref(a), C.byref(b)))
    return a.value, b.value


# ------------------------------------------------------------------------------------------------
# raw C-ABI rendering calls (rt_render_*), used by the sharded multi-GPU path and by tests
# ------------------------------------------------------------------------------------------------
def render_params(width: int, height: int, samples_number: int, max_depth: int, seed: int = 0,
                  shard_count: int = 1, shard_index: int = 0, tile: int = 0) -> RenderParams:
    p = RenderParams()
    p.image = ImageParams(width, height)
    p.samples_number = samples_number
    p.max_depth = max_depth
    p.seed = seed
    p.shard_count = shard_count
    p.shard_index = shard_index
    p.tile_width = tile
    p.tile_height = tile
    return p


_started = {}   # device handle -> (height, width, adaptive) of the last frame started through this module


def _handle_key(dev_scene) -> int:
    return dev_scene.value if isinstance(dev_scene, C.c_void_p) else int(dev_scene)


def render_start(dev_scene, camera: Camera, params: RenderParams) -> None:
    _check(_ffi.core().rt_render_start(dev_scene, C.byref(camera), C.byref(params)))
    _started[_handle_key(dev_scene)] = (params.image.height, params.image.width, False)


def render_start_adaptive(dev_scene, camera: Camera, params: RenderParams, min_samples: int, rel_error: float,
                          abs_error: float = 0.0) -> None:
    """rt_render_start_adaptive: every pixel gets min_samples samples, then doubles its count while the standard error
    of its mean luminance exceeds max(rel_error * |mean|, abs_error), up to params.samples_number.  Each pixel equals
    the render_start frame's pixel at the count it ended with, bit for bit.  Poll / wait deliver the whole frame."""
    ap = _ffi.AdaptiveParams(min_samples, rel_error, abs_error)
    _check(_ffi.core().rt_render_start_adaptive(dev_scene, C.byref(camera), C.byref(params), C.byref(ap)))
    _started[_handle_key(dev_scene)] = (params.image.height, params.image.width, True)


def render_pixel_stats(dev_scene, shape=None):
    """rt_render_pixel_stats of the last completed frame (waits for the frame in flight): counts[h, w] uint32 = samples
    per pixel, moments[h, w, 2] float64 = (Σy, Σy²) of the samples' luminance, or None when the frame was not adaptive.
    shape = (height, width) for a frame not started through render_start / render_start_adaptive."""
    known = _started.get(_handle_key(dev_scene))
    if shape is None:
        if known is None:
            raise ValueError("frame size unknown: pass shape=(height, width)")
        shape = known[:2]
    adaptive = known is not None and known[2]
    h, w = shape
    counts = np.empty((h, w), np.uint32)
    moments = np.empty((h, w, 2), np.float64) if adaptive else None
    _check(_ffi.core().rt_render_pixel_stats(dev_scene, counts.ctypes.data_as(C.c_void_p),
                                             moments.ctypes.data_as(C.c_void_p) if adaptive else None))
    return counts, moments


def standard_error(counts: np.ndarray, moments: np.ndarray) -> np.ndarray:
    """the standard error of each pixel's mean luminance, with the stopping rule's arithmetic (rt_b200.h)"""
    n = counts.astype(np.float64)
    sy, syy = moments[..., 0], moments[..., 1]
    mean = sy / n
    var = np.fmax(0.0, (syy - sy * mean) / (n - 1.0))
    return np.sqrt(var / n)


def render_poll(dev_scene, buffer: Optional[np.ndarray]) -> bool:
    done = C.c_int(0)
    ptr = buffer.ctypes.data_as(C.c_void_p) if buffer is not None else None
    _check(_ffi.core().rt_render_poll(dev_scene, ptr, C.byref(done)))
    return bool(done.value)


def render_wait(dev_scene, buffer: Optional[np.ndarray]) -> None:
    ptr = buffer.ctypes.data_as(C.c_void_p) if buffer is not None else None
    _check(_ffi.core().rt_render_wait(dev_scene, ptr))


def render_set_accumulate(dev_scene, enabled: bool) -> None:
    """progressive accumulation across render_start calls (rt_render_set_accumulate)"""
    _check(_ffi.core().rt_render_set_accumulate(dev_scene, 1 if enabled else 0))


def render_accumulated_samples(dev_scene) -> int:
    n = C.c_uint32(0)
    _check(_ffi.core().rt_render_accumulated_samples(dev_scene, C.byref(n)))
    return n.value


def render_device_result(dev_scene):
    """(device pointer, n) of the shard's tile-packed accumulator: n x 4 doubles (sum r, g, b; samples)."""
    ptr, n = C.c_void_p(), C.c_uint64()
    _check(_ffi.core().rt_render_device_result(dev_scene, C.byref(ptr), C.byref(n)))
    return ptr.value, n.value


def shard_float4_count(params: RenderParams, shard_index: int) -> int:
    return _ffi.core().rt_shard_float4_count(C.byref(params), shard_index)


def assemble_frame(dev_scene, params: RenderParams, shard_ptrs, d_frame_ptr: int, stream: int = 0) -> None:
    arr = (C.c_void_p * len(shard_ptrs))(*shard_ptrs)
    _check(_ffi.core().rt_assemble_frame(dev_scene, C.byref(params), arr, C.c_void_p(d_frame_ptr),
                                         C.c_void_p(stream) if stream else None))


class DevicePointer:
    """Expose a raw device allocation to torch (torch.as_tensor(DevicePointer(...), device='cuda'))
    through __cuda_array_interface__, without copying."""

    def __init__(self, ptr: int, shape, typestr: str = "<f8", owner=None):
        self._owner = owner
        self.__cuda_array_interface__ = {"data": (int(ptr), False), "shape": tuple(shape), "typestr": typestr,
                                         "version": 3, "strides": None}
