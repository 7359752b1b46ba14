"""Step timeline of rank 0 in a data-parallel run + host enqueue cost per step.
usage: torchrun --nproc-per-node N tools/dp_trace.py"""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch, torch.distributed as dist
import ga3c_b200

local = int(os.environ.get("LOCAL_RANK", 0)); rank = int(os.environ.get("RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1))
dev = torch.device("cuda", local); torch.cuda.set_device(dev)
if world > 1:
    dist.init_process_group("nccl", device_id=dev)
tb = 1024
net = ga3c_b200.Network(f"gpu:{local}", "dptrace", 6, max_batch=tb, seed=1)
xs = [(torch.randint(0, 256, (tb, 84 * 84 * 4), device=dev, dtype=torch.int32).float() / 128 - 1).contiguous() for _ in range(3)]
yr = torch.rand(tb, device=dev) * 2 - 1
a = torch.nn.functional.one_hot(torch.randint(0, 6, (tb,), device=dev), 6).float().contiguous()
for i in range(30):
    net.train_device(xs[i % 3], yr, a)
torch.cuda.synchronize()
if world > 1: dist.barrier(device_ids=[local])
# host enqueue cost vs device time over 200 steps
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
torch.cuda.synchronize(); t0 = time.perf_counter(); e0.record()
for i in range(200):
    net.train_device(xs[i % 3], yr, a)
t_enq = time.perf_counter() - t0
e1.record(); torch.cuda.synchronize()
print(f"[rank {rank}] host enqueue {t_enq / 200 * 1e6:.1f} us/step, device {e0.elapsed_time(e1) / 200 * 1e3:.1f} us/step", flush=True)
if world > 1: dist.barrier(device_ids=[local])
for reps in (1, 3):
    torch.cuda.synchronize()
    if world > 1: dist.barrier(device_ids=[local])
    net.trace_begin()
    for i in range(reps):
        net.train_device(xs[i % 3], yr, a)
    rows = net.trace_end()
    if rank == 0:
        print(f"--- {reps} step(s), world {world}")
        for k, v in sorted(rows.items(), key=lambda kv: kv[1][2]):
            print(f"{k:14s} " + " ".join(f"{t:8.1f}" for t in v))
import ctypes as C
from ga3c_b200 import _capi
lib = _capi.load()
torch.cuda.synchronize()
if world > 1: dist.barrier(device_ids=[local])
_capi.check(lib.ga3c_evt_begin(net._h), "evt_begin")
for i in range(2):
    net.train_device(xs[i % 3], yr, a)
buf = (C.c_uint64 * (2 * 16384))(); cnt = C.c_int32()
_capi.check(lib.ga3c_evt_end(net._h, buf, 16384, C.byref(cnt)), "evt_end")
if rank == 0:
    recs = sorted((buf[2 * i], buf[2 * i + 1] >> 32, (buf[2 * i + 1] >> 16) & 0xFFFF, buf[2 * i + 1] & 0xFFFF) for i in range(cnt.value))
    names = {60: "dp_small: launched", 61: "dp_small: dependency satisfied", 62: "dp_small: slabs summed", 66: "dp_small: sums pushed",
             63: "dp_small: every rank's column block arrived", 64: "dp_small: updated"}
    t0 = recs[0][0]
    for t, w, e, arg in recs:
        if e >= 60 and w == 0: print(f"{(t - t0) / 1e3:9.2f} us  {names.get(e, e)} {arg}")
if world > 1: dist.destroy_process_group()
