"""Does DistributedRenderer.render_features deliver the unsharded features frame, bit for bit, for a sequence of frames
whose camera and sample count change from frame to frame?

  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29564 \
      tools/check_distributed_features.py

Every rank renders its tiles; rank 0 compares each assembled frame and its features with rt_render_start_features on
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
w, h, depth, seed = 120, 70, 8, 2024   # (70 rows: clipped border tiles)
sc = rt.Scene.from_file(os.path.join(ROOT, "scenes", "cornell_box.json"), random_spheres_seed=1)
cam = sc.camera()
orbit = api.orbit_cameras(cam, 5)
JOBS = [(cam, 3), (orbit[1], 2), (orbit[3], 1), (cam, 5)]   # (camera, spp)
dr = DistributedRenderer(sc, depth, seed=seed, tile=32, device=lr)
got = [dr.render_features(c, w, h, spp) for c, spp in JOBS]   # back to back
failed = 0
if rank == 0:
    ref_sc = rt.Scene.from_file(os.path.join(ROOT, "scenes", "cornell_box.json"), random_spheres_seed=1)
    hd = ref_sc.device_scene(lr)
    for (c, spp), (frame, feats) in zip(JOBS, got):
        api.render_start_features(hd, c, api.render_params(w, h, spp, depth, seed))
        ref = np.zeros((h, w, 3))
        api.render_wait(hd, ref)
        ref_feats = api.render_features(hd)
        same = np.array_equal(frame, ref) and all(
            feats[k].shape == ref_feats[k].shape and feats[k].tobytes() == ref_feats[k].tobytes() for k in ref_feats)
        failed += int(not same)
        print(f"features, {spp} spp on {world} rank(s): {'identical' if same else 'DIFFERS'}", flush=True)
if world > 1:
    flag = torch.tensor([failed], device="cuda")
    dist.broadcast(flag, 0)
    failed = int(flag[0])
    dist.destroy_process_group()
sys.exit(1 if failed else 0)
