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


def orbit_cameras(camera: Camera, n: int) -> list:
    """n cameras around the scene (a turntable): camera k is `camera` with its position, direction and up rotated about
    the world y axis through the origin by 2*pi*k/n, made by Camera::new with the same focal length and fov"""
    out = []
    for k in range(n):
        a = 2.0 * math.pi * k / n
        c, s = math.cos(a), math.sin(a)
        rot = lambda v: (c * v.x + s * v.z, v.y, c * v.z - s * v.x)
        out.append(camera_new(rot(camera.position), rot(camera.direction), rot(camera.up), camera.focal_length,
                              camera.fov_rad))
    return out


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


def shadow_rays(points: np.ndarray, targets: np.ndarray):
    """rays from points (n, 3) toward targets (n, 3) and the distance of each target: (rays (n, 6), dist (n,)).  The
    direction is Ray::new's unit vector (make_rays) and dist = sqrt((x*x + y*y) + z*z) of targets - points, the same
    length it divides by.  For a shadow ray, pass a t_max a little below dist (e.g. (1 - 1e-9) * dist) to Scene.occluded
    so that the light's own surface at the target does not count."""
    p = np.ascontiguousarray(points, dtype=np.float64).reshape(-1, 3)
    q = np.ascontiguousarray(targets, dtype=np.float64).reshape(-1, 3)
    if p.shape != q.shape:
        raise ValueError(f"points and targets need the same number of rows, got {p.shape[0]} and {q.shape[0]}")
    d = q - p
    dist = np.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1] + d[:, 2] * d[:, 2])
    return make_rays(p, d), dist


def check_t_max(t_max, n: int):
    """occluded's bound: a float (one bound for every ray) or n per-ray bounds as a contiguous (n,) float64 array (numpy,
    or a CUDA torch tensor for occluded_device); returns (scalar, array or None)"""
    if isinstance(t_max, (int, float, np.floating, np.integer)):
        return float(t_max), None
    shape, dtype = tuple(getattr(t_max, "shape", ())), str(getattr(t_max, "dtype", type(t_max).__name__))
    if shape != (n,) or dtype not in ("float64", "torch.float64"):
        raise ValueError(f"t_max must be a float or a ({n},) float64 array, got shape {shape} dtype {dtype}")
    contiguous = t_max.is_contiguous() if hasattr(t_max, "is_contiguous") else t_max.flags["C_CONTIGUOUS"]
    if not contiguous:
        raise ValueError("t_max must be contiguous")
    return math.inf, t_max


SCATTER_OUTPUTS = ("index", "t", "outcome", "color", "scattered")   # rt_scatter_batch's output order


def check_scatter_inputs(rays, keys) -> None:
    """Scene.scatter's inputs: rays a contiguous (n, 6) float64 array and keys a contiguous (n, 2) uint32 array (pixel,
    sample), both numpy or both CUDA torch tensors on one device"""
    is_torch = type(rays).__module__.split(".")[0] == "torch"
    if is_torch != (type(keys).__module__.split(".")[0] == "torch"):
        raise ValueError("rays and keys: both numpy arrays or both torch tensors")
    if is_torch:
        if not (rays.is_cuda and keys.is_cuda):
            raise ValueError("rays and keys: CUDA tensors")
        if keys.device != rays.device:
            raise ValueError(f"keys are on {keys.device}, rays are on {rays.device}")
        contiguous = rays.is_contiguous() and keys.is_contiguous()
    elif not (isinstance(rays, np.ndarray) and isinstance(keys, np.ndarray)):
        raise ValueError("rays and keys: numpy arrays or CUDA torch tensors")
    else:
        contiguous = rays.flags["C_CONTIGUOUS"] and keys.flags["C_CONTIGUOUS"]
    rdt, kdt = str(rays.dtype).replace("torch.", ""), str(keys.dtype).replace("torch.", "")
    if len(rays.shape) != 2 or rays.shape[1] != 6 or rdt != "float64":
        raise ValueError(f"rays: an (n, 6) float64 array, got shape {tuple(rays.shape)} dtype {rdt}")
    if tuple(keys.shape) != (rays.shape[0], 2) or kdt != "uint32":
        raise ValueError(f"keys: an ({rays.shape[0]}, 2) uint32 array, got shape {tuple(keys.shape)} dtype {kdt}")
    if not contiguous:
        raise ValueError("rays and keys must be contiguous")


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

    def set_transforms(self, index, translate, rotate_deg, scale) -> None:
        """Move shapes: shape index[i] gets InversableTransform::new(translate[i], rotate_deg[i], scale[i]) (k x 3 each).
        The description and every device handle this scene has created change together (rth_scene_set_transforms);
        a frame started afterwards on any of them renders the moved shapes."""
        index = np.asarray(index).reshape(-1)
        if index.dtype.kind not in "ui" or (index.size and (index.min() < 0 or index.max() > 0xFFFFFFFF)):
            raise ValueError("set_transforms: shape indices must be integers in [0, 2^32)")
        index = index.astype(np.uint32)
        t, r, s = (np.asarray(a, np.float64).reshape(-1, 3) for a in (translate, rotate_deg, scale))
        if not (len(t) == len(r) == len(s) == index.reshape(-1).shape[0]):
            raise ValueError("set_transforms: index, translate, rotate_deg and scale need one entry per shape")
        rows = [transform(t[k], r[k], s[k]) for k in range(len(t))]
        inv = np.array([x[0] for x in rows]).reshape(-1, 12)
        direct = np.array([x[1] for x in rows]).reshape(-1, 12)
        self.set_transform_rows(index, inv, direct)

    def set_transform_rows(self, index, inverse, direct) -> None:
        """set_transforms with the description's rows 0..2 given directly: index (k,) uint32, inverse and direct (k, 12)
        float64, as api.update_transforms takes them"""
        index, inverse, direct = check_transforms(index, inverse, direct)
        pad = lambda a: np.ascontiguousarray(np.concatenate([a, np.tile([0.0, 0.0, 0.0, 1.0], (len(a), 1))], axis=1))
        inv16, dir16 = pad(inverse), pad(direct)
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        _check(_ffi.host().rth_scene_set_transforms(self._h, len(index), p(index), p(dir16), p(inv16)), host=True)

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

    def occluded(self, rays: np.ndarray, min_t: float = 0.001, max_t=math.inf, mode: int = _ffi.RT_ISECT_FAST,
                 device: Optional[int] = None) -> np.ndarray:
        """any-hit (rt_occluded_batch): is something between min_t and max_t along each ray?  Exactly
        closest_hit(rays, min_t, max_t, RT_ISECT_BRUTE)["index"] != -1, stopping at the first shape that accepts the
        ray.  max_t: a float, or a contiguous (n,) float64 array of per-ray bounds.  Returns an (n,) bool array."""
        rays = np.ascontiguousarray(rays, dtype=np.float64).reshape(-1, 6)
        n = rays.shape[0]
        t_max, per_ray = check_t_max(max_t, n)
        out = np.empty(n, np.uint8)
        p = lambda a: a.ctypes.data_as(C.c_void_p) if a is not None else None
        _check(_ffi.core().rt_occluded_batch(self.device_scene(device), p(rays), n, min_t, t_max, p(per_ray), mode,
                                             p(out)))
        return out.view(np.bool_)

    def scatter(self, rays, keys, level: int, seed: int = 0, min_t: float = 0.001, max_t: float = math.inf,
                mode: int = _ffi.RT_ISECT_FAST, device: Optional[int] = None) -> dict:
        """one segment of ray_color for each ray (rt_scatter_batch): the nearest hit, then what its material does with
        the ray, with the frame's RNG stream of sample keys[i, 1] of pixel keys[i, 0] at its level-th hit.  Returns
        {"index": (n,) int32, "t": (n,) float64, "outcome": (n,) uint8 (RT_BOUNCE_MISS / _SCATTER / _EMIT), "color":
        (n, 3) float64 (sky, attenuation or emission), "scattered": (n, 6) float64 (origin, unit direction)}.
        rays (n, 6) float64 and keys (n, 2) uint32, both contiguous: numpy arrays -> numpy results after the host round
        trip; or CUDA torch tensors on the scene's device -> torch tensors there, queued on torch's current stream
        without a host synchronisation (rt_scatter_batch_device)."""
        check_scatter_inputs(rays, keys)
        n = rays.shape[0]
        if type(rays).__module__.split(".")[0] == "torch":
            import torch
            h = self.device_scene(device)
            if rays.device.index != self._device:
                raise ValueError(f"rays are on {rays.device}, the scene's device is cuda:{self._device}")
            new = lambda shape, dt: torch.empty(shape, dtype=dt, device=rays.device)
            out = {"index": new((n,), torch.int32), "t": new((n,), torch.float64), "outcome": new((n,), torch.uint8),
                   "color": new((n, 3), torch.float64), "scattered": new((n, 6), torch.float64)}
            # torch's default stream is the legacy default stream (handle 0), which the ABI names cudaStreamLegacy = 0x1
            stream = torch.cuda.current_stream(rays.device).cuda_stream or 1
            _check(_ffi.core().rt_scatter_batch_device(h, rays.data_ptr(), keys.data_ptr(), n, level, seed, min_t,
                                                       max_t, mode, *(out[k].data_ptr() for k in SCATTER_OUTPUTS),
                                                       stream))
            return out
        out = {"index": np.empty(n, np.int32), "t": np.empty(n), "outcome": np.empty(n, np.uint8),
               "color": np.empty((n, 3)), "scattered": np.empty((n, 6))}
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        _check(_ffi.core().rt_scatter_batch(self.device_scene(device), p(rays), p(keys), n, level, seed, min_t, max_t,
                                            mode, *(p(out[k]) for k in SCATTER_OUTPUTS)))
        return out

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

    def render_counts(self, camera: Camera, counts: np.ndarray, samples_number: Optional[int] = None) -> np.ndarray:
        """A frame with the caller's sample count per pixel (rt_render_start_counts) on this renderer's devices, depth
        and seed: counts is an (h, w) uint32 map, e.g. the counts render_adaptive returned.  Returns frame[h, w, 3]
        float64; a pixel with count 0 is NaN.  samples_number is the cap the counts are checked against (default: the
        largest count, 1 for an all-zero map)."""
        if getattr(counts, "ndim", 0) != 2:
            raise ValueError("counts: a (height, width) uint32 array")
        height, width = counts.shape
        counts = check_counts(counts, width, height)
        if samples_number is None:
            samples_number = max(int(counts.max(initial=0)), 1)
        if self.devices and len(self.devices) > 1:
            h = self.scene.device_scene_multi(self.devices)
        else:
            h = self.scene.device_scene(self.device)
        render_start_counts(h, camera, render_params(width, height, samples_number, self.depth, self.seed), counts)
        frame = np.zeros((height, width, 3), np.float64)
        render_wait(h, frame)
        return frame

    def render_views(self, cameras, width: int, height: int, samples_number: int) -> np.ndarray:
        """Several views of the scene in one frame (rt_render_start_views) on this renderer's devices, depth and seed:
        returns frames[V, h, w, 3] float64, frames[v] equal to render(cameras[v], width, height, samples_number) bit for
        bit."""
        cameras = check_cameras(cameras)
        if self.devices and len(self.devices) > 1:
            h = self.scene.device_scene_multi(self.devices)
        else:
            h = self.scene.device_scene(self.device)
        render_start_views(h, cameras, render_params(width, height, samples_number, self.depth, self.seed))
        frames = np.zeros((len(cameras), height, width, 3), np.float64)
        render_wait(h, frames)
        return frames

    def render_layers(self, camera: Camera, width: int, height: int, samples_number: int, n_layers: int):
        """A frame with its bounce layers (rt_render_start_layers) on this renderer's devices, depth and seed: returns
        (frame[h, w, 3], layers[n_layers, h, w, 3]) float64.  frame is render(camera, ...) bit for bit; layer b holds the
        radiance of the paths that ended on level b (the last layer: on level n_layers - 1 or deeper), divided by the
        pixel's sample count, so the layers add up to the frame."""
        if self.devices and len(self.devices) > 1:
            h = self.scene.device_scene_multi(self.devices)
        else:
            h = self.scene.device_scene(self.device)
        render_start_layers(h, camera, render_params(width, height, samples_number, self.depth, self.seed), n_layers)
        frame = np.zeros((height, width, 3), np.float64)
        render_wait(h, frame)
        return frame, render_layers(h)

    def render_features(self, camera: Camera, width: int, height: int, samples_number: int):
        """A frame with its first-hit features (rt_render_start_features) on this renderer's devices, depth and seed:
        returns (frame[h, w, 3] float64, features), frame = render(camera, ...) bit for bit and features the dict of
        render_features: albedo, normal, depth, coverage, shape."""
        if self.devices and len(self.devices) > 1:
            h = self.scene.device_scene_multi(self.devices)
        else:
            h = self.scene.device_scene(self.device)
        render_start_features(h, camera, render_params(width, height, samples_number, self.depth, self.seed))
        frame = np.zeros((height, width, 3), np.float64)
        render_wait(h, frame)
        return frame, render_features(h)


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


def transform(translate, rotate_deg, scale):
    """InversableTransform::new: (inverse, direct) rows 0..2 as two float64 arrays of 12, the rows rt_scene_desc holds"""
    direct = np.zeros(16, np.float64)
    inverse = np.zeros(16, np.float64)
    _check(_ffi.host().rth_transform_new(vec3(translate), vec3(rotate_deg), vec3(scale),
                                         direct.ctypes.data_as(C.POINTER(C.c_double)),
                                         inverse.ctypes.data_as(C.POINTER(C.c_double))), host=True)
    return inverse[:12].copy(), direct[:12].copy()


def translated_rows(inverse, direct, shift):
    """the description rows (k, 12) of shapes moved by world-space offsets shift (k, 3), rotation and scale kept:
    T' = translate(shift) o T, so direct's translation column gains shift and inverse's loses M^-1 shift"""
    inverse = np.array(inverse, np.float64).reshape(-1, 3, 4)
    direct = np.array(direct, np.float64).reshape(-1, 3, 4)
    shift = np.asarray(shift, np.float64).reshape(-1, 3)
    inverse[:, :, 3] -= np.einsum("kij,kj->ki", inverse[:, :, :3], shift)
    direct[:, :, 3] += shift
    return inverse.reshape(-1, 12), direct.reshape(-1, 12)


def random_walk(scene: "Scene", index, n_frames: int, step: float, seed: int = 0):
    """n_frames positions of the shapes `index` of `scene` on a seeded random walk in the x-z plane (N(0, step) per
    axis and frame): a list of (index, inverse, direct), the arguments of update_transforms, one per frame"""
    index = np.asarray(index, np.uint32)
    d = scene.desc()
    inv = np.ctypeslib.as_array(d.inverse, shape=(d.n_shapes, 12))[index].copy()
    direct = np.ctypeslib.as_array(d.direct, shape=(d.n_shapes, 12))[index].copy()
    rng = np.random.default_rng(seed)
    frames = []
    for _ in range(n_frames):
        shift = rng.normal(0.0, step, (len(index), 3)) * (1.0, 0.0, 1.0)
        inv, direct = translated_rows(inv, direct, shift)
        frames.append((index, inv, direct))
    return frames


def scene_update(dev_scene, desc: _ffi.SceneDesc) -> None:
    """rt_scene_update: the handle renders `desc` from now on (validated like rt_scene_create; on failure it keeps its
    scene)"""
    _check(_ffi.core().rt_scene_update(dev_scene, C.byref(desc)))


def check_transforms(index, inverse, direct):
    """the arguments of update_transforms as contiguous arrays: index (k,) uint32, inverse and direct (k, 12) float64"""
    index = np.asarray(index)
    inverse = np.asarray(inverse)
    direct = np.asarray(direct)
    if index.ndim != 1 or index.dtype != np.uint32:
        raise ValueError(f"index must be a (k,) uint32 array, got {index.shape} {index.dtype}")
    k = index.shape[0]
    for name, a in (("inverse", inverse), ("direct", direct)):
        if a.shape != (k, 12) or a.dtype != np.float64:
            raise ValueError(f"{name} must be a ({k}, 12) float64 array, got {a.shape} {a.dtype}")
    return (np.ascontiguousarray(index), np.ascontiguousarray(inverse), np.ascontiguousarray(direct))


def update_transforms(dev_scene, index, inverse, direct) -> None:
    """rt_scene_update_transforms: shapes index[i] get inverse rows inverse[i] and direct rows direct[i] (rows 0..2 of
    InversableTransform); the cull tree is refit in place, nothing waits for the device.  This moves the shapes of this
    handle only: for a handle of a Scene (Scene.device_scene) use Scene.set_transforms, which keeps the Scene's
    description and all its handles in step."""
    index, inverse, direct = check_transforms(index, inverse, direct)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    _check(_ffi.core().rt_scene_update_transforms(dev_scene, index.shape[0], p(index), p(inverse), p(direct)))


def occluded_device(dev_scene, rays, out, t_max=math.inf, t_min: float = 0.001, mode: int = _ffi.RT_ISECT_FAST):
    """rt_occluded_batch_device on torch CUDA tensors of the handle's device, queued on torch's current stream without a
    host synchronisation: rays (n, 6) float64, out (n,) uint8 or bool (1 = occluded), t_max a float or an (n,) float64
    tensor, all contiguous.  Returns out."""
    import torch
    if not (rays.is_cuda and rays.dtype == torch.float64 and rays.dim() == 2 and rays.shape[1] == 6
            and rays.is_contiguous()):
        raise ValueError("rays: a contiguous float64 CUDA tensor of shape (n, 6)")
    n = rays.shape[0]
    if not (out.is_cuda and out.dtype in (torch.uint8, torch.bool) and tuple(out.shape) == (n,) and out.is_contiguous()):
        raise ValueError(f"out: a contiguous uint8 or bool CUDA tensor of shape ({n},)")
    t_scalar, per_ray = check_t_max(t_max, n)
    if per_ray is not None and not per_ray.is_cuda:
        raise ValueError("t_max: per-ray bounds must be a CUDA tensor")
    for name, tns in (("out", out), ("t_max", per_ray)):
        if tns is not None and tns.device != rays.device:
            raise ValueError(f"{name} is on {tns.device}, rays are on {rays.device}")
    # torch's default stream is the legacy default stream (handle 0), which the ABI names cudaStreamLegacy = 0x1
    stream = torch.cuda.current_stream(rays.device).cuda_stream or 1
    _check(_ffi.core().rt_occluded_batch_device(dev_scene, rays.data_ptr(), n, t_min, t_scalar,
                                                per_ray.data_ptr() if per_ray is not None else None, mode,
                                                out.data_ptr(), stream))
    return out


MAX_LEVEL = 62   # the deepest level a frame reaches (rt_render_params.max_depth <= 62)


def trace_paths(scene: Scene, rays, keys, depth: int, seed: int = 0, record: bool = False):
    """ray_color (src/renderer/mod.rs:23-45) as a bounce loop over Scene.scatter, in the frame's own arithmetic: the
    throughput starts at (1, 1, 1) and is multiplied forward (beta = beta * color at a scatter), a path ends with
    L = beta * color at a miss or an emission and with L = 0 at a hit on level `depth`, and only the paths still alive
    go to the next level's call.  Ray i is sample keys[i, 1] of pixel keys[i, 0]; fed a frame's primary rays, the
    result averaged by group_means is that frame bit for bit.  rays / keys as Scene.scatter takes them (numpy, or CUDA
    torch tensors: then every level runs on torch's current stream).
    Returns the (n, 3) float32 radiance; with record=True also a list with one dict per level of the paths alive there:
    "ray" (which input ray), "shape", "outcome", "origin", "color" and "beta" (the throughput the path arrives with)."""
    if not 0 <= depth <= MAX_LEVEL:
        raise ValueError(f"depth must be in [0, {MAX_LEVEL}], got {depth}")
    check_scatter_inputs(rays, keys)
    n = rays.shape[0]
    if type(rays).__module__.split(".")[0] == "torch":
        import torch
        full = lambda v: torch.full((n, 3), v, dtype=torch.float64, device=rays.device)
        live = torch.arange(n, device=rays.device)
        where = lambda m: torch.nonzero(m).reshape(-1)
        # (uint32 tensors cannot be gathered on every torch build: the keys are moved as int32)
        ikeys = keys.view(torch.int32)
        take_keys = lambda idx: ikeys[idx].view(torch.uint32)
        to_f32 = lambda a: a.to(torch.float32)
    else:
        full = lambda v: np.full((n, 3), v)
        live = np.arange(n)
        where = np.flatnonzero
        take_keys = lambda idx: keys[idx]
        to_f32 = lambda a: a.astype(np.float32)
    beta, L = full(1.0), full(0.0)
    levels = []
    cur = rays
    for level in range(depth + 1):
        if len(live) == 0:
            break
        out = scene.scatter(cur, keys if level == 0 else take_keys(live), level, seed)
        oc, col, b = out["outcome"], out["color"], beta[live]
        if record:
            levels.append({"ray": live, "shape": out["index"], "outcome": oc, "origin": cur[:, :3], "color": col,
                           "beta": b})
        # a miss ends the path with the sky, an emission with its light; on the last level a hit is black (mod.rs:26-27)
        end = where(oc == _ffi.RT_BOUNCE_MISS) if level == depth else where(oc != _ffi.RT_BOUNCE_SCATTER)
        L[live[end]] = b[end] * col[end]
        if level == depth:
            break
        go = where(oc == _ffi.RT_BOUNCE_SCATTER)
        live = live[go]
        beta[live] = b[go] * col[go]
        cur = out["scattered"][go]
    return (to_f32(L), levels) if record else to_f32(L)


def _philox_uniforms(seed: int, pixel, sample, event: int):
    """the first two doubles of the path RNG's stream (seed; pixel, sample, event): Philox4x32-10 of the counter
    (pixel, sample, event, 0) under the key (seed low, seed high) -- the device's PathRng.next(), twice"""
    m32 = np.uint64(0xFFFFFFFF)
    c0, c1 = pixel.astype(np.uint64), sample.astype(np.uint64)
    c2, c3 = np.full_like(c0, event), np.zeros_like(c0)
    k0, k1 = seed & 0xFFFFFFFF, seed >> 32
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c0, np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ np.uint64(k0), p1 & m32, (p0 >> np.uint64(32)) ^ c3 ^ np.uint64(k1), p0 & m32
        k0, k1 = (k0 + 0x9E3779B9) & 0xFFFFFFFF, (k1 + 0xBB67AE85) & 0xFFFFFFFF
    a = (c1 << np.uint64(32)) | c0
    b = (c3 << np.uint64(32)) | c2
    s53 = 1.0 / 9007199254740992.0
    return (a >> np.uint64(11)).astype(np.float64) * s53, (b >> np.uint64(11)).astype(np.float64) * s53


def primary_rays(camera: Camera, width: int, height: int, pixels, spp: int, seed: int = 0):
    """the frame's own primary rays of `pixels` (indices x + y*width), samples 0 .. spp-1 of each, sample-minor, with
    their keys (pixel, sample): MultisamplerRayCaster::next (src/camera/ray_caster.rs:100-118) with the two draws of
    event 0 of each path's RNG, in the frame's arithmetic.  Returns (rays (n, 6) float64, keys (n, 2) uint32), what
    trace_paths takes to reproduce those pixels of a render_start frame of this camera, size and seed."""
    pix = np.repeat(np.asarray(pixels, np.uint32).reshape(-1), spp)
    smp = np.tile(np.arange(spp, dtype=np.uint32), pix.size // max(spp, 1))
    u, v = _philox_uniforms(seed, pix, smp, 0)
    # MultisamplerRayCaster::new (ray_caster.rs:30-48), as the library computes it on the host
    pos, dirn = camera.position.tuple(), camera.direction.tuple()
    right, up = camera.right.tuple(), camera.up.tuple()
    center = [pos[k] + dirn[k] * camera.focal_length for k in range(3)]
    vw = math.tan(camera.fov_rad / 2.0) * camera.focal_length * 2.0
    vh = vw / (width / height)
    hw, hh = vw / 2.0, vh / 2.0
    left_top = [(center[k] - hw * right[k]) + hh * up[k] for k in range(3)]
    res = vw / width
    x = (pix % width).astype(np.float64) + u
    y = (pix // width).astype(np.float64) + v
    d = np.stack([(left_top[k] + (res * x) * right[k]) - (res * y) * up[k] - pos[k] for k in range(3)], 1)
    ln = np.sqrt((d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2])
    rays = np.empty((pix.size, 6))
    rays[:, :3] = pos
    rays[:, 3:] = d / ln[:, None]
    return rays, np.ascontiguousarray(np.stack([pix, smp], 1))


def group_means(radiance, offsets) -> np.ndarray:
    """the per-group mean of per-ray radiance as trace_pixel_samples_group and the frame take it: group g = rays
    offsets[g] .. offsets[g+1]-1, f64 sums of the float radiance in ray order from 0.0, one division by the group's
    count (an empty group is NaN).  radiance (n, 3) float32 (numpy or torch); returns (G, 3) float64 numpy."""
    if type(radiance).__module__.split(".")[0] == "torch":
        radiance = radiance.cpu().numpy()
    f = np.asarray(radiance, dtype=np.float32).reshape(-1, 3).astype(np.float64)
    off = np.asarray(offsets, dtype=np.int64).reshape(-1)
    if off.size == 0 or off[0] != 0 or off[-1] != f.shape[0] or (np.diff(off) < 0).any():
        raise ValueError("offsets must rise from 0 to len(radiance)")
    count = np.diff(off)
    s = np.zeros((count.size, 3))
    for k in range(int(count.max(initial=0))):   # step k adds ray k of every group that has one: the in-order sums
        m = count > k
        s[m] = s[m] + f[off[:-1][m] + k]
    with np.errstate(invalid="ignore"):
        return s / count[:, None]


def check_counts(counts, width: int, height: int) -> np.ndarray:
    """a sample-count map for a width x height frame: a C-contiguous (height, width) uint32 array"""
    if not isinstance(counts, np.ndarray) or counts.dtype != np.uint32:
        raise ValueError(f"counts: a uint32 numpy array, got {getattr(counts, 'dtype', type(counts).__name__)}")
    if counts.shape != (height, width):
        raise ValueError(f"counts: shape (height, width) = {(height, width)} expected, got {counts.shape}")
    return np.ascontiguousarray(counts)


def render_start_counts(dev_scene, camera: Camera, params: RenderParams, counts: np.ndarray) -> None:
    """rt_render_start_counts: pixel x + y*width gets counts[y, x] samples (0 .. counts-1), at most
    params.samples_number; each pixel equals the render_start frame's pixel at that sample count, bit for bit, and a
    pixel with count 0 is NaN.  counts covers the whole image, also for a shard.  Poll / wait deliver as for
    render_start."""
    counts = check_counts(counts, params.image.width, params.image.height)
    _check(_ffi.core().rt_render_start_counts(dev_scene, C.byref(camera), C.byref(params),
                                              counts.ctypes.data_as(C.c_void_p)))
    _started[_handle_key(dev_scene)] = (params.image.height, params.image.width, False)


def check_cameras(cameras) -> list:
    """the cameras of a views frame: a non-empty sequence of Camera"""
    if isinstance(cameras, Camera):
        raise ValueError("cameras: a sequence of Camera, got a single Camera")
    try:
        cameras = list(cameras)
    except TypeError:
        raise ValueError(f"cameras: a sequence of Camera, got {type(cameras).__name__}") from None
    if not cameras:
        raise ValueError("cameras: at least one Camera")
    for i, c in enumerate(cameras):
        if not isinstance(c, Camera):
            raise ValueError(f"cameras[{i}]: a Camera, got {type(c).__name__}")
    return cameras


def render_start_views(dev_scene, cameras, params: RenderParams) -> None:
    """rt_render_start_views: one frame of len(cameras) views of params.image's size each.  The frame is the stacked
    image (width, len(cameras) * height), view v in rows v*height .. v*height+height-1, so that poll / wait deliver
    buffer[v, y, x] of a (V, h, w, 3) buffer; view v equals render_start of cameras[v] with params, bit for bit.  An
    explicit shard (shard_count > 1) is a shard of the stacked image: size and assemble it with params whose
    image.height is len(cameras) * height."""
    cameras = check_cameras(cameras)
    table = (Camera * len(cameras))(*cameras)
    _check(_ffi.core().rt_render_start_views(dev_scene, table, len(cameras), C.byref(params)))
    _started[_handle_key(dev_scene)] = (len(cameras) * params.image.height, params.image.width, False)


def stacked_params(params: RenderParams, n_views: int) -> RenderParams:
    """the params of the stacked image of a views frame (for shard_float4_count and assemble_frame)"""
    p = RenderParams.from_buffer_copy(params)
    p.image = ImageParams(params.image.width, n_views * params.image.height)
    return p


MAX_LAYERS = MAX_LEVEL + 1   # a layers frame keeps at most one layer per level


def check_n_layers(n_layers) -> int:
    if isinstance(n_layers, bool) or not isinstance(n_layers, (int, np.integer)):
        raise ValueError(f"n_layers: an int, got {type(n_layers).__name__}")
    if not 1 <= n_layers <= MAX_LAYERS:
        raise ValueError(f"n_layers must be in [1, {MAX_LAYERS}], got {n_layers}")
    return int(n_layers)


def render_start_layers(dev_scene, camera: Camera, params: RenderParams, n_layers: int) -> None:
    """rt_render_start_layers: the render_start frame (poll / wait deliver it as for render_start), and with it layer b
    of every pixel = the f64 sum, in sample order, of the radiance of its samples whose path ended on level
    min(level, n_layers - 1) == b, over the pixel's sample count (render_layers)"""
    n_layers = check_n_layers(n_layers)
    _check(_ffi.core().rt_render_start_layers(dev_scene, C.byref(camera), C.byref(params), n_layers))
    _started[_handle_key(dev_scene)] = (params.image.height, params.image.width, False)


def render_layers(dev_scene, device: bool = False, shape=None):
    """rt_render_layers after a completed unsharded layers frame (waits for the frame in flight): layers[L, h, w, 3]
    float64, layer b of pixel (x, y) at [b, y, x].  device=True returns (device pointer, n) of the library's copy on
    the handle's first device instead (n = L * h * w rt_vec3, valid until the next frame starts).  shape = (height,
    width) for a frame not started through render_start_layers."""
    ptr, n = C.c_void_p(), C.c_uint64()
    _check(_ffi.core().rt_render_layers(dev_scene, None, C.byref(ptr), C.byref(n)))
    if device:
        return ptr.value, n.value
    if shape is None:
        known = _started.get(_handle_key(dev_scene))
        if known is None:
            raise ValueError("frame size unknown: pass shape=(height, width)")
        shape = known[:2]
    h, w = shape
    if h * w == 0 or n.value % (h * w):
        raise ValueError(f"shape {shape} does not divide the {n.value} pixels of the layers")
    out = np.empty((n.value // (h * w), h, w, 3), np.float64)
    _check(_ffi.core().rt_render_layers(dev_scene, out.ctypes.data_as(C.c_void_p), None, None))
    return out


def render_device_layers(dev_scene):
    """(device pointer, n) of the shard's layer sums: n = L * shard_float4_count slots of 3 doubles, layer-major, each
    layer in the tile-packed order of render_device_result"""
    ptr, n = C.c_void_p(), C.c_uint64()
    _check(_ffi.core().rt_render_device_layers(dev_scene, C.byref(ptr), C.byref(n)))
    return ptr.value, n.value


def assemble_layers(dev_scene, params: RenderParams, n_layers: int, acc_ptrs, sum_ptrs, d_out_ptr: int,
                    stream: int = 0) -> None:
    """rt_assemble_layers: the gathered accumulators and layer sums of every shard -> L x h x w x 3 layers at
    d_out_ptr, on `stream` (0: the library's stream)"""
    if len(acc_ptrs) != len(sum_ptrs):
        raise ValueError("one accumulator and one layer-sum buffer per shard")
    accs = (C.c_void_p * len(acc_ptrs))(*acc_ptrs)
    sums = (C.c_void_p * len(sum_ptrs))(*sum_ptrs)
    _check(_ffi.core().rt_assemble_layers(dev_scene, C.byref(params), n_layers, accs, sums, C.c_void_p(d_out_ptr),
                                          C.c_void_p(stream) if stream else None))


def path_levels(record, n: int) -> np.ndarray:
    """the level that ended each of the n paths of trace_paths(..., record=True): the last level whose record lists the
    path (record[k]["ray"]).  Returns (n,) int32; -1 for a path no level lists (none, when every path is recorded)."""
    levels = np.full(n, -1, np.int32)
    for k, rec in enumerate(record):
        ray = rec["ray"]
        if type(ray).__module__.split(".")[0] == "torch":
            ray = ray.cpu().numpy()
        levels[np.asarray(ray, np.int64)] = k
    return levels


def layer_means(radiance, levels, offsets, n_layers: int) -> np.ndarray:
    """the layers of groups of paths as the layers frame takes them: layer b of group g = the f64 sum of the float
    radiance of its rays (offsets[g] .. offsets[g+1]-1) whose level has min(level, n_layers - 1) == b, in ray order
    from +0.0, over the group's ray count (an empty group is NaN).  radiance (n, 3) float32 (numpy or torch), levels
    (n,) integers in [0, 62]; returns (n_layers, G, 3) float64."""
    n_layers = check_n_layers(n_layers)
    if type(radiance).__module__.split(".")[0] == "torch":
        radiance = radiance.cpu().numpy()
    f = np.asarray(radiance, dtype=np.float32).reshape(-1, 3).astype(np.float64)
    lv = np.asarray(levels).reshape(-1)
    if lv.shape[0] != f.shape[0] or not np.issubdtype(lv.dtype, np.integer):
        raise ValueError("levels: one integer level per ray")
    if lv.size and (lv.min() < 0 or lv.max() > MAX_LEVEL):
        raise ValueError(f"levels must be in [0, {MAX_LEVEL}]")
    off = np.asarray(offsets, dtype=np.int64).reshape(-1)
    if off.size == 0 or off[0] != 0 or off[-1] != f.shape[0] or (np.diff(off) < 0).any():
        raise ValueError("offsets must rise from 0 to len(radiance)")
    count = np.diff(off)
    b = np.minimum(lv, n_layers - 1)
    s = np.zeros((n_layers, count.size, 3))
    for k in range(int(count.max(initial=0))):   # step k adds ray k of every group that has one, to its layer
        g = np.flatnonzero(count > k)
        r = off[:-1][g] + k
        s[b[r], g] = s[b[r], g] + f[r]
    with np.errstate(invalid="ignore"):
        return s / count[None, :, None]


FEATURE_NAMES = ("albedo", "normal", "depth", "coverage", "shape")
FEATURE_SUMS_DTYPE = np.dtype([("albedo", "<f8", 3), ("normal", "<f8", 3), ("depth", "<f8"), ("hits", "<f8"),
                               ("shape", "<i4"), ("pad", "<u4")])   # rt_feature_sums, 72 bytes


def render_start_features(dev_scene, camera: Camera, params: RenderParams) -> None:
    """rt_render_start_features: the render_start frame (poll / wait deliver it as for render_start), and with it the
    first-hit features of every pixel (render_features): albedo, normal, depth, coverage and shape"""
    _check(_ffi.core().rt_render_start_features(dev_scene, C.byref(camera), C.byref(params)))
    _started[_handle_key(dev_scene)] = (params.image.height, params.image.width, False)


def _feature_planes(ptrs: dict) -> _ffi.FeaturePlanes:
    unknown = set(ptrs) - set(FEATURE_NAMES)
    if unknown:
        raise ValueError(f"unknown feature planes {sorted(unknown)}; the planes are {FEATURE_NAMES}")
    return _ffi.FeaturePlanes(*(C.c_void_p(ptrs[k]) if ptrs.get(k) else None for k in FEATURE_NAMES))


def render_features(dev_scene, device: bool = False, shape=None) -> dict:
    """rt_render_features after a completed unsharded features frame (waits for the frame in flight): {"albedo": (h, w, 3),
    "normal": (h, w, 3), "depth": (h, w), "coverage": (h, w) float64, "shape": (h, w) int32} numpy arrays, pixel (x, y)
    at [y, x].  device=True returns the device pointers of the library's planes on the handle's first device instead
    (valid until the next frame starts).  shape = (height, width) for a frame not started through this module."""
    if device:
        planes = _ffi.FeaturePlanes()
        _check(_ffi.core().rt_render_features(dev_scene, None, C.byref(planes)))
        return {k: getattr(planes, k) for k in FEATURE_NAMES}
    if shape is None:
        known = _started.get(_handle_key(dev_scene))
        if known is None:
            raise ValueError("frame size unknown: pass shape=(height, width)")
        shape = known[:2]
    h, w = shape
    out = {"albedo": np.empty((h, w, 3)), "normal": np.empty((h, w, 3)), "depth": np.empty((h, w)),
           "coverage": np.empty((h, w)), "shape": np.empty((h, w), np.int32)}
    host = _feature_planes({k: v.ctypes.data for k, v in out.items()})
    _check(_ffi.core().rt_render_features(dev_scene, C.byref(host), None))
    return out


def render_device_features(dev_scene):
    """(device pointer, n) of the shard's feature sums: n rt_feature_sums (FEATURE_SUMS_DTYPE, 72 bytes) in the
    tile-packed order of render_device_result"""
    ptr, n = C.c_void_p(), C.c_uint64()
    _check(_ffi.core().rt_render_device_features(dev_scene, C.byref(ptr), C.byref(n)))
    return ptr.value, n.value


def assemble_features(dev_scene, params: RenderParams, sum_ptrs, out_ptrs: dict, stream: int = 0) -> None:
    """rt_assemble_features: the gathered feature sums of every shard -> the planes at out_ptrs (a dict of device
    pointers by FEATURE_NAMES; a missing or zero one is not written), on `stream` (0: the library's stream)"""
    sums = (C.c_void_p * len(sum_ptrs))(*sum_ptrs)
    _check(_ffi.core().rt_assemble_features(dev_scene, C.byref(params), sums, C.byref(_feature_planes(out_ptrs)),
                                            C.c_void_p(stream) if stream else None))


def feature_means(index, t, normal, color, offsets) -> dict:
    """the first-hit features of groups of camera rays as the features frame takes them: group g = rays offsets[g] ..
    offsets[g+1]-1 (a pixel's samples in sample order), index / t / normal their nearest hit (Scene.closest_hit), color
    their level-0 colour (Scene.scatter(level=0)["color"]).  f64 sums in ray order from +0.0: albedo = Σ color / n,
    normal = Σ normal / n (a miss adds zero), depth = Σ t over the hits / hits (+inf without a hit), coverage = hits / n,
    shape = the index of the group's first ray (-1 for an empty group); an empty group's means are NaN.  Returns
    {"albedo": (G, 3), "normal": (G, 3), "depth": (G,), "coverage": (G,) float64, "shape": (G,) int32}."""
    idx = np.asarray(index).reshape(-1)
    if not np.issubdtype(idx.dtype, np.integer):
        raise ValueError("index: one integer shape index per ray")
    n = idx.shape[0]
    tt = np.asarray(t, dtype=np.float64).reshape(-1)
    nrm = np.asarray(normal, dtype=np.float64)
    col = np.asarray(color, dtype=np.float64)
    if tt.shape != (n,) or nrm.shape != (n, 3) or col.shape != (n, 3):
        raise ValueError("t (n,), normal (n, 3) and color (n, 3): one entry per ray")
    off = np.asarray(offsets, dtype=np.int64).reshape(-1)
    if off.size == 0 or off[0] != 0 or off[-1] != n or (np.diff(off) < 0).any():
        raise ValueError("offsets must rise from 0 to len(index)")
    count = np.diff(off)
    hit = idx >= 0
    nrm = np.where(hit[:, None], nrm, 0.0)
    a, nm = np.zeros((count.size, 3)), np.zeros((count.size, 3))
    d, hits = np.zeros(count.size), np.zeros(count.size)
    for k in range(int(count.max(initial=0))):   # step k adds ray k of every group that has one: the in-order sums
        g = np.flatnonzero(count > k)
        r = off[:-1][g] + k
        a[g] = a[g] + col[r]
        nm[g] = nm[g] + nrm[r]
        gh, rh = g[hit[r]], r[hit[r]]
        d[gh] = d[gh] + tt[rh]
        hits[gh] = hits[gh] + 1.0
    shape = np.full(count.size, -1, np.int32)
    shape[count > 0] = idx[off[:-1][count > 0]]
    with np.errstate(invalid="ignore", divide="ignore"):
        return {"albedo": a / count[:, None], "normal": nm / count[:, None],
                "depth": np.where(hits > 0, d / np.maximum(hits, 1.0), np.inf), "coverage": hits / count,
                "shape": shape}


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
