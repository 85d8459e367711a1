"""N-GPU data-parallel check of the occupancy-grid engine (run under torchrun): the all-reduced
gradient of the ray-sharded step equals the single-GPU gradient of the same global batch, and after
a grid update every rank holds the same grid.
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \
        --master-port 29711 tools/dp_check_occgrid.py
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from fsnerf_b200 import parallel, synthetic as syn  # noqa: E402
from fsnerf_b200.engine import HotPath  # noqa: E402

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
G = 2048
H = W = 64
AABB = [-1.5] * 3 + [1.5] * 3
poses, imgs, focal = syn.make_views(4, H, W, seed=42)
rng = np.random.default_rng(0)
ids = rng.permutation(4 * H * W)[:G]
o = np.concatenate([syn.camera_rays(p, H, W, focal)[0].reshape(-1, 3) for p in poses])[ids]
d = np.concatenate([syn.camera_rays(p, H, W, focal)[1].reshape(-1, 3) for p in poses])[ids]
gt = imgs.reshape(-1, 3)[ids]
u = rng.random(G, dtype=np.float32)
cu = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)  # noqa: E731


def engine(world_size=None):
    hp = HotPath(sampler="occgrid", roi_aabb=AABB, grid_resolution=128, device=dev, world_size=world_size)
    sd = hp.state_dict(0)
    sd["sigma.bias"] += 3.0  # dense enough for the visibility filter to matter
    hp.load_state_dict(0, sd)
    hp.update_grid(0)
    return hp


a, b = parallel.shard_range(G, rank, world)
hp = engine()
ls = hp.train_step(cu(o[a:b]), cu(d[a:b]), cu(gt[a:b]), u_strat=cu(u[a:b]), global_rays=G, apply_update=False)
ls = ls.clone()
dist.all_reduce(ls)
ok = True
if rank == 0:
    hp1 = engine(world_size=1)
    ls1 = hp1.train_step(cu(o), cu(d), cu(gt), u_strat=cu(u), global_rays=G, apply_update=False)
    rel = ((hp.grads - hp1.grads).norm() / hp1.grads.norm()).item()
    dl = (ls - ls1).abs().max().item() / ls1.abs().max().item()
    print(f"occgrid dp{world} vs single GPU: grad rel err {rel:.3e}, loss rel err {dl:.3e}")
    ok = rel < 1e-3 and dl < 1e-5
# one more step with the update: k = 1 steps Adam, then an update at k = 16 on the fresh weights
hp.train_step(cu(o[a:b]), cu(d[a:b]), cu(gt[a:b]), global_rays=G)
hp.update_grid(16)
grids = [torch.empty_like(hp.estimator.occs) for _ in range(world)]
dist.all_gather(grids, hp.estimator.occs)
params = [torch.empty_like(hp.params) for _ in range(world)]
dist.all_gather(params, hp.params)
same = all(torch.equal(g, grids[0]) for g in grids) and all(torch.equal(p, params[0]) for p in params)
if rank == 0:
    print(f"occgrid dp{world}: params and grids identical on every rank: {same}")
ok = ok and same
dist.barrier()
dist.destroy_process_group()
sys.exit(0 if ok else 1)
