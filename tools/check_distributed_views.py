"""Does DistributedRenderer.render_views deliver the unsharded views frame, bit for bit, for camera sets that change
from frame to frame?

  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29562 \
      tools/check_distributed_views.py

Every rank passes the same cameras; rank 0 compares each assembled set of views with rt_render_start of every camera on
one device of its own.  Exit code 1 on a deviation."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np, torch, torch.distributed as dist
import rs_pathtracing_b200 as rt
from rs_pathtracing_b200 import api
from rs_pathtracing_b200.distributed import DistributedRenderer

rank, world, lr = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
torch.cuda.set_device(lr)
if world > 1:
    dist.init_process_group("nccl", device_id=torch.device(f"cuda:{lr}"))
w, h, spp, depth, seed = 120, 70, 3, 8, 2024   # (70 rows: the 32x32 tiles straddle the views)
sc = rt.Scene.from_file(os.path.join(ROOT, "scenes", "cornell_box.json"), random_spheres_seed=1)
cam = sc.camera()
SETS = [api.orbit_cameras(cam, 5), [cam], api.orbit_cameras(cam, 8)[::-1]]
dr = DistributedRenderer(sc, depth, seed=seed, tile=32, device=lr)
frames = []
for cams in SETS:   # back to back
    f = dr.render_views(cams, w, h, spp)
    frames.append(None if f is None else f.copy())
failed = 0
if rank == 0:
    ref_sc = rt.Scene.from_file(os.path.join(ROOT, "scenes", "cornell_box.json"), random_spheres_seed=1)
    hd = ref_sc.device_scene(lr)
    for i, cams in enumerate(SETS):
        ref = np.zeros((len(cams), h, w, 3))
        for v, c in enumerate(cams):
            api.render_start(hd, c, api.render_params(w, h, spp, depth, seed))
            api.render_wait(hd, ref[v])
        same = frames[i].shape == ref.shape and np.array_equal(frames[i], ref)
        failed += int(not same)
        print(f"{len(cams)} views on {world} rank(s): {'identical' if same else 'DIFFERS'}", flush=True)
if world > 1:
    flag = torch.tensor([failed], device="cuda")
    dist.broadcast(flag, 0)
    failed = int(flag[0])
    dist.destroy_process_group()
sys.exit(1 if failed else 0)
