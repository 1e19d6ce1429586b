"""Does a pipelined moving-object sequence of DistributedRenderer equal frame-by-frame renders on fresh handles?

  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29566 \
      tools/check_distributed_scene_update.py

Every rank renders the same sequence through render_jobs_device, two frames in flight on two handles, where each job
carries a fifth element (index, inverse, direct) that moves some of the random spheres (api.random_walk; some jobs move
nothing).  Rank 0 compares every assembled frame with rt_render_start on a handle freshly created from the description
edited up to that job, and checks that the scene's description holds the last positions afterwards.  Then
DistributedRenderer.update_transforms moves the spheres back and one more frame must equal the unedited scene's.
Exit code 1 on a deviation."""
import ctypes as C, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np, torch, torch.distributed as dist
import rs_pathtracing_b200 as rt
from rs_pathtracing_b200 import _ffi, api
from rs_pathtracing_b200.distributed import DistributedRenderer

rank, world, lr = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
torch.cuda.set_device(lr)
if world > 1:
    dist.init_process_group("nccl", device_id=torch.device(f"cuda:{lr}"))
w, h, spp, depth, seed = 96, 64, 2, 8, 77
path = os.path.join(ROOT, "scenes", "spheres.json")
sc = rt.Scene.from_file(path, random_spheres_seed=1)
cam = sc.camera()
n_file = rt.Scene.from_file(path, add_random_spheres=False).shape_count
d0 = sc.desc()
inv0 = np.ctypeslib.as_array(d0.inverse, shape=(d0.n_shapes, 12)).copy()
dir0 = np.ctypeslib.as_array(d0.direct, shape=(d0.n_shapes, 12)).copy()
walk = api.random_walk(sc, np.arange(n_file, n_file + 40), 6, 0.3, seed=5)
edits = [walk[0], None, walk[1], walk[2], None, walk[3], walk[4], walk[5]]
jobs = [(cam, w, h, spp, e) for e in edits]
dr = DistributedRenderer(sc, depth, seed=seed, tile=32, device=lr)
frames = []
dr.render_jobs_device(jobs, on_frame=lambda i, f: frames.append(f.cpu().numpy().copy()))
failed = 0
if rank == 0:
    inv, direct = inv0.copy(), dir0.copy()
    for i, e in enumerate(edits):
        if e is not None:
            inv[e[0]], direct[e[0]] = e[1], e[2]
        d = sc.desc()
        d.inverse = inv.ctypes.data_as(C.POINTER(C.c_double))
        d.direct = direct.ctypes.data_as(C.POINTER(C.c_double))
        hd = C.c_void_p()
        api._check(_ffi.core().rt_scene_create(C.byref(d), lr, C.byref(hd)))
        api.render_start(hd, cam, api.render_params(w, h, spp, depth, seed))
        ref = np.empty((h, w, 3))
        api.render_wait(hd, ref)
        _ffi.core().rt_scene_destroy(hd)
        same = np.array_equal(frames[i], ref)
        failed += int(not same)
        print(f"job {i} ({'moves' if e is not None else 'no edit'}) on {world} rank(s): {'identical' if same else 'DIFFERS'}",
              flush=True)
    d = sc.desc()
    in_step = np.array_equal(np.ctypeslib.as_array(d.inverse, shape=(d.n_shapes, 12)), inv)
    failed += int(not in_step)
    print(f"scene description after the sequence: {'in step' if in_step else 'STALE'}", flush=True)
# back to the start through update_transforms (the scene, its handle and the second handle)
moved = np.arange(n_file, n_file + 40, dtype=np.uint32)
dr.update_transforms(moved, inv0[moved], dir0[moved])
last = []
dr.render_jobs_device([(cam, w, h, spp), (cam, w, h, spp)], on_frame=lambda i, f: last.append(f.cpu().numpy().copy()))
if rank == 0:
    ref_sc = rt.Scene.from_file(path, random_spheres_seed=1)
    hd = ref_sc.device_scene(lr)
    api.render_start(hd, cam, api.render_params(w, h, spp, depth, seed))
    ref = np.empty((h, w, 3))
    api.render_wait(hd, ref)
    for i, f in enumerate(last):
        same = np.array_equal(f, ref)
        failed += int(not same)
        print(f"after update_transforms, frame {i}: {'identical' if same else 'DIFFERS'}", flush=True)
if world > 1:
    flag = torch.tensor([failed], device="cuda")
    dist.broadcast(flag, 0)
    failed = int(flag[0])
    dist.destroy_process_group()
print(f"deviating frames {failed}", flush=True)
sys.exit(1 if failed else 0)
