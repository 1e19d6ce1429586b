"""Does DistributedRenderer.render_layers deliver the unsharded layers frame, bit for bit, for a sequence of frames whose
camera, layer count and sample count change from frame to frame?

  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29563 \
      tools/check_distributed_layers.py

Every rank renders its tiles; rank 0 compares each assembled frame and its layers with rt_render_start_layers on one
device of its own.  Exit code 1 on a deviation."""
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
w, h, depth, seed = 120, 70, 8, 2024   # (70 rows: clipped border tiles)
sc = rt.Scene.from_file(os.path.join(ROOT, "scenes", "cornell_box.json"), random_spheres_seed=1)
cam = sc.camera()
orbit = api.orbit_cameras(cam, 5)
JOBS = [(cam, 3, 4), (orbit[1], 2, 63), (orbit[3], 1, 1), (cam, 5, 9)]   # (camera, spp, n_layers)
dr = DistributedRenderer(sc, depth, seed=seed, tile=32, device=lr)
got = [dr.render_layers(c, w, h, spp, n) for c, spp, n in JOBS]   # back to back
failed = 0
if rank == 0:
    ref_sc = rt.Scene.from_file(os.path.join(ROOT, "scenes", "cornell_box.json"), random_spheres_seed=1)
    hd = ref_sc.device_scene(lr)
    for (c, spp, n), (frame, layers) in zip(JOBS, got):
        api.render_start_layers(hd, c, api.render_params(w, h, spp, depth, seed), n)
        ref = np.zeros((h, w, 3))
        api.render_wait(hd, ref)
        ref_layers = api.render_layers(hd)
        same = np.array_equal(frame, ref) and layers.shape == ref_layers.shape and \
            layers.tobytes() == ref_layers.tobytes()
        failed += int(not same)
        print(f"{n} layers, {spp} spp on {world} rank(s): {'identical' if same else 'DIFFERS'}", flush=True)
if world > 1:
    flag = torch.tensor([failed], device="cuda")
    dist.broadcast(flag, 0)
    failed = int(flag[0])
    dist.destroy_process_group()
sys.exit(1 if failed else 0)
