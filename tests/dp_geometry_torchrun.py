"""Test infrastructure (launched by tests/test_gpu_geometry.py on boxes with >= 2 GPUs, or by hand with torchrun): the
data-parallel step at a geometry other than 84x84x4, where Network uses dp_mode 'nccl'.  Every rank trains on its row shard of
one global batch; afterwards the replicas hold bit-identical weights that match the geometry oracle's steps on the whole batch.
Prints 'DP_GEOMETRY OK' on rank 0."""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import numpy as np
import torch
import torch.distributed as dist

rank, local, world = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
import ga3c_b200
from ga3c_b200.dataparallel import shard_rows
from oracle import oracle_np as onp        # checker only

HWC = (42, 42, 4)


class Cfg(ga3c_b200.Config):
    IMAGE_HEIGHT, IMAGE_WIDTH, STACKED_FRAMES = HWC


g = onp.Geometry(*HWC)
B = 16 * world
rng = np.random.default_rng(4242)
params = onp.init_params(rng, 6, geom=g)
net = ga3c_b200.Network(f"gpu:{local}", "dpgeo", 6, config=Cfg, max_batch=64)
assert net.dp_mode == "nccl", net.dp_mode
net.set_variables(params)
ref = {k: v.astype(np.float64) for k, v in params.items()}
ms, mom = onp.rmsprop_init(ref)
for step in range(3):
    x = onp.normalise(onp.synth_frames_u8(rng, B, geom=g))
    y_r, a = onp.synth_targets(rng, B, 6)
    lo, hi = shard_rows(B, rank, world)
    net.train(x[lo:hi], y_r[lo:hi], a[lo:hi], None, None, 0)
    _, grads = onp.loss_and_grads({k: v.astype(np.float32) for k, v in ref.items()}, x, y_r, a, geom=g, quant="bf16",
                               beta=net.beta)
    ref, ms, mom = onp.rmsprop_update(ref, grads, ms, mom, lr=net.learning_rate, dtype=np.float64)
got = net.get_variables()
flat = torch.from_numpy(np.concatenate([got[k].ravel() for k in sorted(got)])).cuda()
gathered = [torch.zeros_like(flat) for _ in range(world)]
dist.all_gather(gathered, flat)
identical = all(torch.equal(gathered[0], t) for t in gathered)
worst = max(float(np.abs(got[k] - ref[k]).max()) for k in got)
if rank == 0:
    print(f"replicas identical: {identical}; max |w - oracle| after 3 steps: {worst:.3e}")
    assert identical and worst <= 1e-5, (identical, worst)
    print("DP_GEOMETRY OK")
dist.barrier()
dist.destroy_process_group()
