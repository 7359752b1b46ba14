"""Predict and train throughput of the conv network at several input geometries (Config.IMAGE_HEIGHT, IMAGE_WIDTH,
STACKED_FRAMES): 84x84x4 runs the specialised trunk, every other geometry the generic one (conv_gen.cu).  Device-resident inputs
rotated through a ring larger than the 126 MB L2; each figure is the median of >= 100 calls after >= 20 warm-up calls, timed
with CUDA events.  Per-kernel times come from ga3c_timing_* in a separate pass.  The roofline fractions compare the measured time
with the least time of the algorithm's bytes at 7.7 TB/s and of its FLOPs at 2,250 TFLOP/s (data-sheet figures of one B200 at
1,000 W, never reached; computed below from the shapes, independent of the implementation).
usage: python tools/geometry_bench.py [tag]   -> profiles/<tag>_geometry_bench.json"""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import ga3c_b200

GEOMETRIES = [(84, 84, 4), (84, 84, 1), (84, 84, 3), (42, 42, 4), (105, 80, 4), (100, 100, 2), (8, 8, 1), (128, 128, 4)]
PREDICT_B, TRAIN_B, A = (128, 1024, 4096), 1024, 6
L2, HBM, MMA = 126 * 2 ** 20, 7.7e12, 2.25e15
WARMUP, CALLS = 20, 100


def sizes(h, w, c):
    h1, w1 = -(-h // 4), -(-w // 4)
    h2, w2 = -(-h1 // 2), -(-w1 // 2)
    return h1 * w1, h2 * w2, h2 * w2 * 32


def algo_bytes(hwc, b, train):
    """Bytes the computation needs at the least, whatever the implementation: the frames (fp32), p and v, and the weights read
    once (dense1/w as its bf16 copy); train also reads y_r and a and updates the fp32 weights and RMSProp ms in place."""
    h, w, c = hwc
    k = sizes(h, w, c)[2]
    small = 64 * c * 16 + 16 + 256 * 32 + 32 + 256 + 257 * (1 + A)
    weights = k * 256 * 2 + small * 4
    if not train:
        return b * (h * w * c * 4 + (A + 1) * 4) + weights
    arena = k * 256 + small
    return b * (h * w * c * 4 + (A + 1) * 4) + weights + 4 * arena * 4


def algo_flops(hwc, b, train):
    """Multiply-adds x 2 of the three GEMM layers (the heads are negligible); train: forward, data gradient (not for conv11,
    whose input needs none) and weight gradient."""
    h, w, c = hwc
    p1, p2, k = sizes(h, w, c)
    c11, c12, d1 = 2 * p1 * 64 * c * 16, 2 * p2 * 256 * 32, 2 * k * 256
    return b * ((2 * c11 + 3 * c12 + 3 * d1) if train else (c11 + c12 + d1))


def bounds(hwc, b, train, ms):
    """Share of the HBM bound (algorithmic bytes / 7.7 TB/s) and of the compute bound (algorithmic FLOPs / 2,250 TFLOP/s dense
    bf16) in the measured time; `bound` names the larger of the two least times."""
    t_hbm, t_mma = algo_bytes(hwc, b, train) / HBM, algo_flops(hwc, b, train) / MMA
    return {"hbm_roofline_frac": round(t_hbm / (ms * 1e-3), 4), "compute_roofline_frac": round(t_mma / (ms * 1e-3), 4),
            "bound": "hbm" if t_hbm >= t_mma else "compute"}


def config(hwc):
    class Cfg(ga3c_b200.Config):
        pass
    Cfg.IMAGE_HEIGHT, Cfg.IMAGE_WIDTH, Cfg.STACKED_FRAMES = hwc
    return Cfg


def ring(state_dim, b):
    n = max(2, -(-int(1.5 * L2) // (b * state_dim * 4)) + 1)
    return [(torch.randint(0, 256, (b, state_dim), device="cuda", dtype=torch.int32).float() / 128 - 1).contiguous()
            for _ in range(n)]


def timed(fn, n_ring):
    st = torch.cuda.current_stream()
    for i in range(WARMUP):
        fn(i % n_ring)
    torch.cuda.synchronize()
    times = []
    for i in range(CALLS):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        fn(i % n_ring)
        e1.record(st)
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    return float(np.median(times))


def kernel_times(net, fn, n):
    net.kernel_timing(4096)
    for i in range(n):
        fn(i)
    torch.cuda.synchronize()
    out = {k: round(1e3 * ms / cnt, 2) for k, (ms, cnt) in net.kernel_times().items()}      # us per launch
    net.kernel_timing(0)                     # the next timed pass runs without the event brackets
    return out


def main():
    tag = sys.argv[1] if len(sys.argv) > 1 else "dev"
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    out = {"gpu": q or torch.cuda.get_device_name(0), "hbm_peak_bytes_per_s": HBM, "bf16_peak_flops": MMA, "calls": CALLS,
           "warmup": WARMUP, "geometries": []}
    for hwc in GEOMETRIES:
        sd = hwc[0] * hwc[1] * hwc[2]
        net = ga3c_b200.Network("gpu:0", "geobench", A, sd, config=config(hwc), max_batch=max(PREDICT_B), seed=1)
        row = {"geometry": list(hwc), "path": "specialised" if hwc == (84, 84, 4) else "generic", "dense1_k": sizes(*hwc)[2],
               "predict": {}, "train": {}}
        for b in PREDICT_B:
            xs = ring(sd, b)
            p = torch.empty((b, A), device="cuda")
            v = torch.empty((b,), device="cuda")
            fn = lambda i: net.predict_device(xs[i % len(xs)], p, v)      # noqa: E731
            ms = timed(fn, len(xs))
            row["predict"][b] = {"ms": round(ms, 4), "frames_per_s": round(b / ms * 1e3), **bounds(hwc, b, False, ms),
                                 "kernel_us": kernel_times(net, fn, 20)}
            del xs
        b = TRAIN_B
        xs = ring(sd, b)
        yr = torch.rand(b, device="cuda") * 2 - 1
        a = torch.nn.functional.one_hot(torch.randint(0, A, (b,), device="cuda"), A).float().contiguous()
        fn = lambda i: net.train_device(xs[i % len(xs)], yr, a)      # noqa: E731
        ms = timed(fn, len(xs))
        row["train"][b] = {"ms": round(ms, 4), "frames_per_s": round(b / ms * 1e3), **bounds(hwc, b, True, ms),
                           "kernel_us": kernel_times(net, fn, 20)}
        del xs, net
        torch.cuda.empty_cache()
        out["geometries"].append(row)
        print(json.dumps(row), flush=True)
    os.makedirs("profiles", exist_ok=True)
    path = os.path.join("profiles", f"{tag}_geometry_bench.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    print(path, out["gpu"])


if __name__ == "__main__":
    main()
