"""What one Network.log costs at B = 1024 (float32 frames) against the 1000 train steps of its interval
(Config.TENSORBOARD_UPDATE_FREQUENCY; Server.py:149-150), on one GPU.

    python tools/log_bench.py [--batch 1024] [--calls 25] [--steps 1000] [--out FILE]

Reports, in one JSON line (also written to --out):
  - the median wall time of Network.log over --calls calls after warm-up (frames handed over as a pageable numpy array, as
    the reference's trainer does; the event file goes to a temporary directory), and of Network.histograms alone;
  - the histogram kernels' own time (kernel_times()["histograms"], CUDA events) and the bytes they read over it, as a share of
    the 6546.6 GB/s measured HBM read rate;
  - the host alternative: download the weights and the n1 / n2 / d1 workspaces, predict p and v, and run the numpy
    histograms (oracle/histogram_np.py) over them;
  - 1000 back-to-back train steps on device-resident tensors, and log's share of them (target: <= 10 %).
The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
HBM_READ_GBS = 6546.6          # measured HBM read rate of a B200 (SURVEY.md, BASELINE.md)


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        return r.stdout.strip().splitlines()[0] if r.returncode == 0 else "unknown"
    except (OSError, subprocess.SubprocessError, IndexError):
        return "unknown"


def histogram_bytes(net, b: int) -> int:
    """Bytes the histogram kernel reads: every variable (fp32), the live chunks of n1 (bf16, 441 x 16 per frame: the borders of
    its Blk2 layout are not loaded), n2 (bf16), d1 (fp32), v and p (fp32)."""
    weights = sum(int(np.prod(s)) for _, s in net._table.values())
    return 4 * weights + b * (441 * 16 * 2 + 3872 * 2 + 256 * 4 + 4 + 4 * net.num_actions)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--calls", type=int, default=25)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import ga3c_b200
    from oracle import histogram_np as oh
    from oracle import oracle_np as onp

    b = args.batch
    rng = np.random.default_rng(0)
    x = onp.synth_frames(rng, b)
    y_r, a = onp.synth_targets(rng, b)
    net = ga3c_b200.Network("gpu:0", "log_bench", 6, max_batch=b, seed=1)
    dev = torch.device("cuda", 0)
    dx, dyr, da = (torch.from_numpy(t).to(dev) for t in (x, y_r, a))
    res = {"card": card(), "batch": b, "frames": "float32"}

    # train steps first: log then reports on trained weights and activations, as in a run
    for _ in range(50):
        net.train_device(dx, dyr, da)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        net.train_device(dx, dyr, da)
    torch.cuda.synchronize()
    train_ms = (time.perf_counter() - t0) * 1e3
    res["train_steps"] = args.steps
    res["train_ms"] = round(train_ms, 3)
    res["step_ms"] = round(train_ms / args.steps, 5)

    cwd = os.getcwd()
    with tempfile.TemporaryDirectory() as tmp:
        os.chdir(tmp)
        try:
            for i in range(3):
                net.log(x, y_r, a, i)
            times = []
            for i in range(args.calls):
                t0 = time.perf_counter()
                net.log(x, y_r, a, 1000 * (i + 1))
                times.append((time.perf_counter() - t0) * 1e3)
        finally:
            os.chdir(cwd)
    res["log_calls"] = args.calls
    res["log_ms_median"] = round(statistics.median(times), 3)
    res["log_ms_min"] = round(min(times), 3)
    times = []
    for _ in range(args.calls):
        t0 = time.perf_counter()
        net.histograms(x, y_r, a)
        times.append((time.perf_counter() - t0) * 1e3)
    res["histograms_call_ms_median"] = round(statistics.median(times), 3)

    net.kernel_timing(1024)
    net.kernel_times()
    n_k = 20
    for _ in range(n_k):
        net.histograms(x, y_r, a)
    kt = net.kernel_times()
    net.kernel_timing(0)
    ms, launches = kt["histograms"]
    kernel_us = ms / n_k * 1e3
    nbytes = histogram_bytes(net, b)
    res["histogram_kernels_us"] = round(kernel_us, 2)
    res["histogram_launches_per_call"] = launches // n_k
    res["histogram_bytes"] = nbytes
    res["histogram_hbm_share"] = round(nbytes / (HBM_READ_GBS * 1e9) / (kernel_us * 1e-6), 3)
    res["histogram_values"] = int(sum(int(np.prod(s)) for _, s in net._table.values()) + b * (7056 + 3872 + 256 + 1 + 6))

    times = []
    for _ in range(3):
        t0 = time.perf_counter()
        w = net.get_variables()
        n1, n2, d1 = net.workspace(0), net.workspace(1), net.workspace(2)
        p, v = net.predict_p_and_v(x)
        for name, t in w.items():
            oh.histogram(t, name)
        for t in (n1, n2, d1, v, p):
            oh.histogram(t)
        times.append((time.perf_counter() - t0) * 1e3)
    res["host_alternative_ms_median"] = round(statistics.median(times), 1)

    res["log_share_of_interval"] = round(res["log_ms_median"] / train_ms, 4)
    res["target_share"] = 0.10
    res["meets_target"] = res["log_share_of_interval"] <= 0.10
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
