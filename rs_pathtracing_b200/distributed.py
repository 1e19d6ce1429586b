"""One process per GPU: interleaved-tile sharding of a frame with a single NCCL gather.

torch / torch.distributed are plumbing only (process group, device buffers for the gather); every
pixel is produced by the CUDA core through the C ABI (rt_render_start with shard_count/shard_index,
rt_render_device_result, rt_assemble_frame).  Tile k (row-major, 32x32 by default) belongs to rank
k % world_size; the RNG is keyed by (pixel, sample, event), so the assembled frame does not depend on
the number of GPUs -- bit for bit: the accumulators exchanged are the f64 sums themselves.

A single-process alternative needs no torch at all: GpuRenderer(scene, ..., devices=[0, 1, ...]) drives every GPU of
the box through one handle of the C ABI (rt_scene_create_multi, peer copies instead of NCCL).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np

from . import api
from ._ffi import Camera

CUDA_STREAM_LEGACY = 0x1   # cudaStreamLegacy (driver_types.h): explicit handle of the legacy default stream


def owned_pixel_coords(width: int, height: int, tile: int, world: int, shard: int):
    """Host mirror of ShardMap::pixel_of (csrc/rt_core.cu): the pixels shard `shard` owns, in its
    tile-packed "owned order" (tile k -> shard k % world; tiles numbered row-major with row ty rotated by ty
    positions, so that a shard owns diagonals rather than columns of tiles when tiles_x is a multiple of world;
    row-major inside a tile, border tiles padded to tile*tile).  Returns (x, y, valid) int arrays of length
    rt_shard_float4_count."""
    if world == 1:   # whole image: one "tile" per row, owned order == x + y*width
        tw, th, skew = width, 1, 0
    else:
        tw = th = tile
        skew = 1
    tiles_x, tiles_y = (width + tw - 1) // tw, (height + th - 1) // th
    ks = np.arange(shard, tiles_x * tiles_y, world)
    ty = ks // tiles_x
    tx = (ks % tiles_x + (ty % tiles_x) * skew) % tiles_x
    r = np.arange(tw * th)
    x = (tx[:, None] * tw + r[None, :] % tw).reshape(-1)
    y = (ty[:, None] * th + r[None, :] // tw).reshape(-1)
    return x, y, (x < width) & (y < height)


def exchange_to_rank0(dist, mine, counts, rank: int, world: int, bufs=None):
    """The one exchange of a frame: every rank's tile-packed accumulator (4 doubles per pixel: f64 sums of r, g, b and
    the sample count, so that the assembled frame is the unsharded one bit for bit) to rank 0 (grouped
    send/recv: shard sizes can differ by one tile, so this is not dist.gather).  Returns the list of the
    `world` shard tensors on rank 0, None elsewhere.  Backend-agnostic (NCCL on GPUs, gloo in the CPU tests)."""
    import torch
    if world == 1:
        return [mine]
    ops = []
    if rank == 0:
        if bufs is None or [b.shape[0] for b in bufs] != list(counts):
            bufs = [torch.empty((c,) + tuple(mine.shape[1:]), dtype=torch.float64, device=mine.device) for c in counts]
        bufs[0].copy_(mine)
        for s in range(1, world):
            ops.append(dist.P2POp(dist.irecv, bufs[s], s))
    else:
        ops.append(dist.P2POp(dist.isend, mine, 0))
    if ops:
        for req in dist.batch_isend_irecv(ops):
            req.wait()
    return bufs if rank == 0 else None


def assemble_host(shards, width: int, height: int, tile: int, world: int) -> np.ndarray:
    """numpy restatement of k_assemble: gathered tile-packed (n, 4) shards -> (h, w, 3) mean radiance"""
    frame = np.zeros((height, width, 3), dtype=np.float64)
    for s, buf in enumerate(shards):
        b = np.asarray(buf, dtype=np.float64)
        x, y, ok = owned_pixel_coords(width, height, tile, world, s)
        frame[y[ok], x[ok]] = b[ok, :3] / b[ok, 3:4]
    return frame


class DistributedRenderer:
    """Renderer-trait-shaped front end for N ranks.  Every rank constructs it with the same scene and
    calls render(); rank 0 returns the full frame (numpy, h x w x 3 float64), the others None."""

    def __init__(self, scene: api.Scene, depth: int, seed: int = 0, tile: int = 32, device: Optional[int] = None):
        import torch
        import torch.distributed as dist

        self.torch, self.dist = torch, dist
        self.rank = dist.get_rank() if dist.is_initialized() else 0
        self.world = dist.get_world_size() if dist.is_initialized() else 1
        self.device = torch.cuda.current_device() if device is None else device
        self.scene, self.depth, self.seed, self.tile = scene, depth, seed, tile
        self.dev_scene = scene.device_scene(self.device)
        self._gather_bufs = None
        self._frame = None
        self._host = None
        self._exchanged = None   # event on torch's stream: the previous frame's accumulator has been read
        # pipelined sequences (render_jobs_device): two staging copies of the shard's accumulator, so that the NEXT
        # frame can start rendering while this one is still being exchanged and assembled
        self._stage = [None, None]
        self._stage_ready = [None, None]   # event on the copy stream: the staging copy is complete
        self._stage_free = [None, None]    # event on torch's stream: the exchange has read the staging buffer
        self._stage_k = 0
        self._copy_stream = None
        self._host2 = [None, None]
        self._dev_scene_b = None           # a second rt_scene on the same device: two frames of a sequence in flight
        self._layer_bufs = None            # rank 0: the gathered layer sums of layers frames
        self._feature_bufs = None          # rank 0: the gathered feature sums of features frames

    def _params(self, w, h, spp, shard):
        return api.render_params(w, h, spp, self.depth, self.seed, self.world, shard, tile=self.tile)

    def render_device(self, camera: Camera, width: int, height: int, samples_number: int, counts=None):
        """Render this rank's tiles, gather, assemble on rank 0.  Returns the device frame tensor on
        rank 0 (h x w x 3 float64), None elsewhere.  No host synchronisation besides NCCL's own.
        counts: an (h, w) uint32 sample-count map (rt_render_start_counts; samples_number is then the cap), the WHOLE
        map on every rank; the assembled frame is the unsharded counts frame, bit for bit."""
        if counts is None:
            start = lambda p: api.render_start(self.dev_scene, camera, p)
        else:
            start = lambda p: api.render_start_counts(self.dev_scene, camera, p, counts)
        return self._render_shard(start, width, height, samples_number)

    def render_views_device(self, cameras, width: int, height: int, samples_number: int):
        """render_device for several views in one frame (rt_render_start_views): every rank renders its tiles of the
        stacked image (width, V * height) and passes the same cameras.  Returns the device frames on rank 0
        (V x h x w x 3 float64, view v equal to render_device(cameras[v], ...) bit for bit), None elsewhere."""
        cameras = api.check_cameras(cameras)
        view = self._params(width, height, samples_number, self.rank)
        frame = self._render_shard(lambda p: api.render_start_views(self.dev_scene, cameras, view),
                                   width, len(cameras) * height, samples_number)
        return None if frame is None else frame.view(len(cameras), height, width, 3)

    def render_layers_device(self, camera: Camera, width: int, height: int, samples_number: int, n_layers: int):
        """render_device of a layers frame (rt_render_start_layers): every rank renders its tiles, and its layer sums
        travel to rank 0 in one more exchange.  Returns (frame h x w x 3, layers n_layers x h x w x 3) float64 device
        tensors on rank 0, each equal to the unsharded layers frame's bit for bit, None elsewhere."""
        n_layers = api.check_n_layers(n_layers)
        return self._render_shard(lambda p: api.render_start_layers(self.dev_scene, camera, p, n_layers),
                                  width, height, samples_number, n_layers)

    def render_features_device(self, camera: Camera, width: int, height: int, samples_number: int):
        """render_device of a features frame (rt_render_start_features): every rank renders its tiles, and its feature
        sums (72 bytes per owned pixel) travel to rank 0 in one more exchange.  Returns (frame h x w x 3 float64,
        features) on rank 0 -- features a dict of device tensors as api.render_features gives them: albedo, normal
        (h, w, 3), depth, coverage (h, w) float64, shape (h, w) int32 -- each equal to the unsharded features frame's
        bit for bit, None elsewhere."""
        return self._render_shard(lambda p: api.render_start_features(self.dev_scene, camera, p),
                                  width, height, samples_number, features=True)

    def _render_shard(self, start, width: int, height: int, samples_number: int, n_layers: int = 0,
                      features: bool = False):
        """start(params) this rank's shard of a width x height frame, gather, assemble on rank 0 (n_layers > 0: a
        layers frame, whose layers are gathered and assembled too: (frame, layers) on rank 0; features: a features
        frame, (frame, features) on rank 0)"""
        torch, dist = self.torch, self.dist
        p = self._params(width, height, samples_number, self.rank)
        # The library renders on its own non-blocking streams, the exchange runs on torch's / NCCL's: the
        # orderings between the two are explicit.  (1) This frame's k_resolve overwrites the accumulator the
        # previous frame's send (rank 0: copy) reads, so that read must be over before the frame starts.
        if self._exchanged is not None:
            self._exchanged.synchronize()
        start(p)
        ptr, n = api.render_device_result(self.dev_scene)   # waits for this shard's kernels
        mine = torch.as_tensor(api.DevicePointer(ptr, (n, 4), "<f8", owner=self), device=f"cuda:{self.device}")
        counts = [api.shard_float4_count(p, s) for s in range(self.world)]
        # one exchange per frame: every rank's tile-packed accumulator to rank 0 over NVLink
        shards = exchange_to_rank0(dist, mine, counts, self.rank, self.world, self._gather_bufs)
        layer_shards = None
        if n_layers:   # the second exchange: every rank's layer sums, n_layers slots of 3 doubles per owned pixel
            lptr, ln = api.render_device_layers(self.dev_scene)
            mine_l = torch.as_tensor(api.DevicePointer(lptr, (ln, 3), "<f8", owner=self), device=f"cuda:{self.device}")
            layer_shards = exchange_to_rank0(dist, mine_l, [n_layers * c for c in counts], self.rank, self.world,
                                             self._layer_bufs)
        feature_shards = None
        if features:   # the second exchange: every rank's feature sums, 72 bytes (moved as 9 doubles) per owned pixel
            fptr, fn = api.render_device_features(self.dev_scene)
            mine_f = torch.as_tensor(api.DevicePointer(fptr, (fn, 9), "<f8", owner=self), device=f"cuda:{self.device}")
            feature_shards = exchange_to_rank0(dist, mine_f, counts, self.rank, self.world, self._feature_bufs)
        if self._exchanged is None:
            self._exchanged = torch.cuda.Event()
        self._exchanged.record()   # (the current stream waits for the NCCL work: req.wait() in exchange_to_rank0)
        if shards is None:
            return None
        if self.world > 1:
            self._gather_bufs = shards
            if n_layers:
                self._layer_bufs = layer_shards
            if features:
                self._feature_bufs = feature_shards
        if self._frame is None or tuple(self._frame.shape) != (height, width, 3):
            self._frame = torch.empty((height, width, 3), dtype=torch.float64, device=mine.device)
        # (2) k_assemble must run after the receives, i.e. on torch's current stream, and the host copy of
        # render() after k_assemble.  torch's default stream has the handle 0, which rt_assemble_frame reads as
        # "the library's stream" (unordered against the NCCL receives: shards arrived after the frame had been
        # assembled from the previous frame's buffers); cudaStreamLegacy (0x1) names that stream explicitly.
        api.assemble_frame(self.dev_scene, self._params(width, height, samples_number, 0),
                           [int(s.data_ptr()) for s in shards], int(self._frame.data_ptr()),
                           stream=int(torch.cuda.current_stream().cuda_stream) or CUDA_STREAM_LEGACY)
        if n_layers:
            layers = torch.empty((n_layers, height, width, 3), dtype=torch.float64, device=mine.device)
            api.assemble_layers(self.dev_scene, self._params(width, height, samples_number, 0), n_layers,
                                [int(s.data_ptr()) for s in shards], [int(s.data_ptr()) for s in layer_shards],
                                int(layers.data_ptr()),
                                stream=int(torch.cuda.current_stream().cuda_stream) or CUDA_STREAM_LEGACY)
        if features:
            new = lambda shape, dt: torch.empty(shape, dtype=dt, device=mine.device)
            feats = {"albedo": new((height, width, 3), torch.float64), "normal": new((height, width, 3), torch.float64),
                     "depth": new((height, width), torch.float64), "coverage": new((height, width), torch.float64),
                     "shape": new((height, width), torch.int32)}
            api.assemble_features(self.dev_scene, self._params(width, height, samples_number, 0),
                                  [int(s.data_ptr()) for s in feature_shards],
                                  {k: int(v.data_ptr()) for k, v in feats.items()},
                                  stream=int(torch.cuda.current_stream().cuda_stream) or CUDA_STREAM_LEGACY)
        self._exchanged.record()   # rank 0's own accumulator is read by k_assemble when it is the only shard
        if features:
            return self._frame, feats
        return (self._frame, layers) if n_layers else self._frame

    # ---- pipelined sequences: frame n's exchange and assembly overlap frame n+1's render ---------------------------
    def _exchange_assemble(self, mine, width, height, samples_number):
        """the exchange + rank 0's k_assemble of render_device, on torch's current stream, reading `mine`"""
        torch, dist = self.torch, self.dist
        p = self._params(width, height, samples_number, self.rank)
        counts = [api.shard_float4_count(p, s) for s in range(self.world)]
        shards = exchange_to_rank0(dist, mine, counts, self.rank, self.world, self._gather_bufs)
        if shards is None:
            return None
        if self.world > 1:
            self._gather_bufs = shards
        if self._frame is None or tuple(self._frame.shape) != (height, width, 3):
            self._frame = torch.empty((height, width, 3), dtype=torch.float64, device=mine.device)
        api.assemble_frame(self.dev_scene, self._params(width, height, samples_number, 0),
                           [int(s.data_ptr()) for s in shards], int(self._frame.data_ptr()),
                           stream=int(torch.cuda.current_stream().cuda_stream) or CUDA_STREAM_LEGACY)
        return self._frame

    def update_transforms(self, index, inverse, direct):
        """Move shapes (api.update_transforms' arguments) in the scene and in both handles of this renderer: the Scene's
        description and every handle it created (Scene.set_transform_rows), and the second handle of the pipelined
        sequences.  Frames started afterwards render the moved shapes."""
        index, inverse, direct = api.check_transforms(index, inverse, direct)
        self.scene.set_transform_rows(index, inverse, direct)
        if self._dev_scene_b is not None:
            api.update_transforms(self._dev_scene_b, index, inverse, direct)

    def render_jobs_device(self, jobs, on_frame=None, on_rendered=None):
        """A SEQUENCE of frames, pipelined: jobs = [(camera, width, height, samples_number), ...].  A job may carry a
        fifth element (index, inverse, direct), the arguments of update_transforms: the shapes move from that frame on.
        The edit is applied to the handle that renders the job just before the job starts, and to the other handle
        before its next job, so a moving-object sequence keeps two frames in flight; once the sequence is done the
        scene and both handles hold the last position of every moved shape.  While frame n's
        accumulators travel to rank 0 and are assembled there, every rank already renders frame n+1 (two frames are in
        flight on two handles of the same device): the serial tail of render_device (host wait -> NCCL send/recv ->
        k_assemble, about 1 ms whatever the frame) and the drain of a frame's last batches disappear from every step
        but the last.  Each frame is still a complete frame on rank 0: on_frame(i, device_frame) is called
        there right after frame i's k_assemble has been ENQUEUED on torch's current stream (consume it on that
        stream, or copy it: the next frame's assembly overwrites it); on_rendered(i) is called on every rank when
        its shard of frame i has finished rendering.  Returns the last device frame (rank 0) / None.

        What makes the overlap safe: the shard's accumulator is copied (device to device, a few microseconds) to one
        of two staging buffers as soon as the shard is complete, and the host waits for THAT copy -- not for the
        exchange -- before it starts the next frame, whose k_resolve overwrites the accumulator.  The exchange reads
        the staging buffer; a staging buffer is rewritten two frames later, after an event says its exchange is
        over."""
        torch = self.torch
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(device=self.device)
        if self._exchanged is not None:     # a preceding render_device(): its send may still read the accumulator
            self._exchanged.synchronize()
        jobs = list(jobs)
        # TWO frames in flight: frame n+1 is already on the device (second handle = its own streams, queues and
        # accumulator) when frame n completes, so the drain of a frame's last batches -- the thin deep bounce levels
        # overlap with nothing -- and the host's turn-around between two frames are filled with the next frame's work.
        handles = [self.dev_scene, self._second_handle()] if len(jobs) > 1 else [self.dev_scene]
        edits = [api.check_transforms(*job[4]) if len(job) > 4 and job[4] is not None else None for job in jobs]
        applied = [0] * len(handles)   # jobs whose edits each handle has received (edits are absolute rows, so in order)

        def start(j):
            hnd = j % len(handles)
            for e in edits[applied[hnd]:j + 1]:
                if e is not None:
                    api.update_transforms(handles[hnd], *e)
            applied[hnd] = j + 1
            cam, w, h, spp = jobs[j][:4]
            api.render_start(handles[hnd], cam, self._params(w, h, spp, self.rank))

        frame = None
        for i in range(min(len(handles), len(jobs))):
            start(i)
        for i, job in enumerate(jobs):
            cam, w, h, spp = job[:4]
            hnd = handles[i % len(handles)]
            ptr, n = api.render_device_result(hnd)   # host: this shard's kernels are done
            if on_rendered is not None:
                on_rendered(i)
            mine = torch.as_tensor(api.DevicePointer(ptr, (n, 4), "<f8", owner=self), device=f"cuda:{self.device}")
            k = self._stage_k = (self._stage_k + 1) % 2
            if self._stage[k] is None or tuple(self._stage[k].shape) != (n, 4):
                self._stage[k] = torch.empty((n, 4), dtype=torch.float64, device=mine.device)
            cs = self._copy_stream
            if self._stage_free[k] is not None:
                cs.wait_event(self._stage_free[k])
            with torch.cuda.stream(cs):
                self._stage[k].copy_(mine)
                if self._stage_ready[k] is None:
                    self._stage_ready[k] = torch.cuda.Event()
                self._stage_ready[k].record(cs)
            self._stage_ready[k].synchronize()                  # host: this handle's accumulator may be overwritten now
            nxt = i + len(handles)
            if nxt < len(jobs):
                start(nxt)
            torch.cuda.current_stream().wait_event(self._stage_ready[k])
            frame = self._exchange_assemble(self._stage[k], w, h, spp)
            if self._stage_free[k] is None:
                self._stage_free[k] = torch.cuda.Event()
            self._stage_free[k].record()
            if frame is not None and on_frame is not None:
                on_frame(i, frame)
        # the last position of every moved shape, into the scene's description (and its handles) and the other handle
        last = {}
        for e in edits:
            if e is not None:
                for k, s in enumerate(e[0]):
                    last[int(s)] = (e[1][k], e[2][k])
        if last:
            index = np.array(sorted(last), np.uint32)
            inverse = np.array([last[s][0] for s in index])
            direct = np.array([last[s][1] for s in index])
            self.scene.set_transform_rows(index, inverse, direct)
            for hnd in handles[1:]:
                api.update_transforms(hnd, index, inverse, direct)
        return frame

    def _second_handle(self):
        if self._dev_scene_b is None:
            from . import _ffi
            h = C.c_void_p()
            d = self.scene.desc()
            api._check(_ffi.core().rt_scene_create(C.byref(d), self.device, C.byref(h)))
            self._dev_scene_b = h
        return self._dev_scene_b

    def __del__(self):
        try:
            if self._dev_scene_b is not None:
                from . import _ffi
                _ffi.core().rt_scene_destroy(self._dev_scene_b)
                self._dev_scene_b = None
        except Exception:
            pass

    def render_many_device(self, camera: Camera, width: int, height: int, samples_number: int, count: int,
                           on_frame=None, on_rendered=None):
        return self.render_jobs_device([(camera, width, height, samples_number)] * count, on_frame, on_rendered)

    def render_jobs(self, jobs, keep: bool = False):
        """render_jobs_device with every frame copied to pinned host memory inside the pipeline (two host buffers,
        asynchronous copies on torch's stream).  Returns the list of host frames when `keep` (copies), else the last
        frame (a view of a pinned buffer, valid until the next call); None on the other ranks."""
        torch = self.torch
        out, events = [], []

        def to_host(i, frame):
            b = i % 2
            if self._host2[b] is None or tuple(self._host2[b].shape) != tuple(frame.shape):
                self._host2[b] = torch.empty(frame.shape, dtype=frame.dtype, pin_memory=True)
            if keep and len(events) >= 2:            # the buffer is about to be reused: take frame i-2 out first
                events[i - 2].synchronize()
                out.append(self._host2[b].numpy().copy())
            self._host2[b].copy_(frame, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record()
            events.append(ev)

        jobs = list(jobs)
        last = self.render_jobs_device(jobs, on_frame=to_host)
        if last is None:
            return None
        torch.cuda.current_stream().synchronize()
        if not keep:
            return self._host2[(len(jobs) - 1) % 2].numpy()
        for i in range(max(len(jobs) - 2, 0), len(jobs)):
            out.append(self._host2[i % 2].numpy().copy())
        return out

    def render(self, camera: Camera, width: int, height: int, samples_number: int, counts=None) -> Optional[np.ndarray]:
        return self._to_host(self.render_device(camera, width, height, samples_number, counts=counts))

    def render_views(self, cameras, width: int, height: int, samples_number: int) -> Optional[np.ndarray]:
        """render_views_device with the frames copied to the host on rank 0: (V, h, w, 3) float64, None elsewhere"""
        return self._to_host(self.render_views_device(cameras, width, height, samples_number))

    def render_layers(self, camera: Camera, width: int, height: int, samples_number: int, n_layers: int):
        """render_layers_device with both copied to the host on rank 0: (frame (h, w, 3), layers (L, h, w, 3)) float64
        numpy arrays of their own, None elsewhere"""
        out = self.render_layers_device(camera, width, height, samples_number, n_layers)
        if out is None:
            return None
        frame, layers = out
        return frame.cpu().numpy(), layers.cpu().numpy()

    def render_features(self, camera: Camera, width: int, height: int, samples_number: int):
        """render_features_device with everything copied to the host on rank 0: (frame (h, w, 3) float64, features dict
        of numpy arrays), arrays of their own, None elsewhere"""
        out = self.render_features_device(camera, width, height, samples_number)
        if out is None:
            return None
        frame, feats = out
        return frame.cpu().numpy(), {k: v.cpu().numpy() for k, v in feats.items()}

    def _to_host(self, frame):
        if frame is None:
            return None
        torch = self.torch
        if self._host is None or tuple(self._host.shape) != tuple(frame.shape):
            self._host = torch.empty(frame.shape, dtype=frame.dtype, pin_memory=True)
        self._host.copy_(frame, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        # (a view of the renderer's pinned buffer: valid until the next render(); copy it to keep it)
        return self._host.numpy()
