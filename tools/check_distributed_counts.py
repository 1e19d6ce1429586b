"""Does DistributedRenderer with a sample-count map deliver the unsharded counts frame, bit for bit, for maps that change
from frame to frame?

  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29561 \
      tools/check_distributed_counts.py

Every rank passes the whole map; rank 0 compares each assembled frame with rt_render_start_counts on one device of its
own (NaN where the count is 0).  Exit code 1 on a deviation."""
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
w, h, depth, seed = 200, 130, 8, 2024
rng = np.random.default_rng(17)
MAPS = [rng.integers(0, 17, (h, w)).astype(np.uint32), np.full((h, w), 3, np.uint32),
        np.where(rng.random((h, w)) < 0.5, 0, 40).astype(np.uint32)]
sc = rt.Scene.from_file(os.path.join(ROOT, "scenes", "cornell_box.json"), random_spheres_seed=1)
cam = sc.camera()
dr = DistributedRenderer(sc, depth, seed=seed, tile=32, device=lr)
frames = []
for counts in MAPS:   # back to back
    f = dr.render(cam, w, h, int(counts.max()), counts=counts)
    frames.append(None if f is None else f.copy())
failed = 0
if rank == 0:
    ref_sc = rt.Scene.from_file(os.path.join(ROOT, "scenes", "cornell_box.json"), random_spheres_seed=1)
    hd = ref_sc.device_scene(lr)
    for i, counts in enumerate(MAPS):
        ref = np.zeros((h, w, 3))
        api.render_start_counts(hd, cam, api.render_params(w, h, int(counts.max()), depth, seed), counts)
        api.render_wait(hd, ref)
        same = np.array_equal(frames[i], ref, equal_nan=True)
        failed += int(not same)
        print(f"counts map {i} on {world} rank(s): {'identical' if same else 'DIFFERS'}", flush=True)
if world > 1:
    flag = torch.tensor([failed], device="cuda")
    dist.broadcast(flag, 0)
    failed = int(flag[0])
    dist.destroy_process_group()
sys.exit(1 if failed else 0)
