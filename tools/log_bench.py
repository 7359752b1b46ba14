"""What one Network.log costs against the 1000 train steps of its interval (Config.TENSORBOARD_UPDATE_FREQUENCY;
Server.py:149-150), on one GPU.

    python tools/log_bench.py [--net conv|fork_vp|discrate] [--batch B] [--calls 25] [--steps 1000] [--out FILE]

--net conv (the default; B = 1024, float32 frames) reports, in one JSON line (also written to --out):
  - the median wall time of Network.log over --calls calls after warm-up (frames handed over as a pageable numpy array, as
    the reference's trainer does; the event file goes to a temporary directory), and of Network.histograms alone;
  - the histogram kernels' own time (kernel_times()["histograms"], CUDA events) and the bytes they read over it, as a share of
    the 6546.6 GB/s measured HBM read rate;
  - the host alternative: download the weights and the n1 / n2 / d1 workspaces, predict p and v, and run the numpy
    histograms (oracle/histogram_np.py) over them;
  - 1000 back-to-back train steps on device-resident tensors, and log's share of them (target: <= 10 %).
--net fork_vp (the fork's NetworkVP, Pendulum: S = 3, A = 1) and --net discrate (NetworkVP_discrate, CartPole: S = 4, A = 2,
Config.DENSE_LAYERS) report the same quantities at B = 1024 and B = 65,536 (or at --batch), one entry per batch in "runs";
the host alternative there downloads the weights and the layer outputs.
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


def measure(net, x, y_r, a, dev, args, res, n_bytes, n_values, host_alternative):
    """Adds to res: back-to-back train steps on the device tensors `dev`, the median Network.log and Network.histograms
    call on the host arrays x, y_r, a, the histogram kernels' own time and bytes, and the host alternative."""
    import torch
    # train steps first: log then reports on trained weights and activations, as in a run
    for _ in range(50):
        net.train_device(*dev)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        net.train_device(*dev)
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
    res["histogram_kernels_us"] = round(kernel_us, 2)
    res["histogram_launches_per_call"] = launches // n_k
    res["histogram_bytes"] = n_bytes
    res["histogram_hbm_share"] = round(n_bytes / (HBM_READ_GBS * 1e9) / (kernel_us * 1e-6), 3)
    res["histogram_values"] = n_values

    times = []
    for _ in range(3):
        t0 = time.perf_counter()
        host_alternative()
        times.append((time.perf_counter() - t0) * 1e3)
    res["host_alternative_ms_median"] = round(statistics.median(times), 1)

    res["log_share_of_interval"] = round(res["log_ms_median"] / train_ms, 4)
    res["target_share"] = 0.10
    res["meets_target"] = res["log_share_of_interval"] <= 0.10
    return res


def conv(args):
    import torch
    import ga3c_b200
    from oracle import histogram_np as oh
    from oracle import oracle_np as onp

    b = args.batch or 1024
    rng = np.random.default_rng(0)
    x = onp.synth_frames(rng, b)
    y_r, a = onp.synth_targets(rng, b)
    net = ga3c_b200.Network("gpu:0", "log_bench", 6, max_batch=b, seed=1)
    dev = torch.device("cuda", 0)
    dx, dyr, da = (torch.from_numpy(t).to(dev) for t in (x, y_r, a))

    def host_alternative():
        w = net.get_variables()
        n1, n2, d1 = net.workspace(0), net.workspace(1), net.workspace(2)
        p, v = net.predict_p_and_v(x)
        for name, t in w.items():
            oh.histogram(t, name)
        for t in (n1, n2, d1, v, p):
            oh.histogram(t)

    values = int(sum(int(np.prod(s)) for _, s in net._table.values()) + b * (7056 + 3872 + 256 + 1 + 6))
    res = {"card": card(), "batch": b, "frames": "float32"}
    return measure(net, x, y_r, a, (dx, dyr, da), args, res, histogram_bytes(net, b), values, host_alternative)


def mlp(args):
    import torch
    from ga3c_b200 import mlp_network
    from oracle import histogram_np as oh
    from oracle import oracle_mlp as om

    kind = args.net
    s, n_act = (3, 1) if kind == "fork_vp" else (4, 2)          # Pendulum / CartPole
    cls = mlp_network.NetworkVP if kind == "fork_vp" else mlp_network.NetworkVP_discrate
    n_layers = len(om.layers_of(kind))
    out = {"card": card(), "net": kind, "state_dim": s, "num_actions": n_act, "runs": []}
    for b in ([args.batch] if args.batch else [1024, 65536]):
        rng = np.random.default_rng(0)
        x = rng.uniform(-1, 1, size=(b, s)).astype(np.float32)
        y_r = rng.uniform(-1, 1, size=b).astype(np.float32)
        a = (rng.uniform(-1, 1, size=(b, n_act)) if kind == "fork_vp"
             else np.eye(n_act)[rng.integers(0, n_act, size=b)]).astype(np.float32)
        net = cls("gpu:0", "logbench", n_act, s, max_batch=b, seed=1)
        dev = torch.device("cuda", 0)
        dx, dyr, da = (torch.from_numpy(t).to(dev) for t in (x, y_r, a))

        def host_alternative():
            w = net.get_variables()
            acts = [net.workspace(0, l, b) for l in range(n_layers)]
            p, v = net.predict_p_and_v(x)
            for name, t in w.items():
                oh.histogram(t, name)
            for t in acts + [v, p]:
                oh.histogram(t)

        # every value ga3c_mlp_histograms reads is fp32: the variables, the live layers' outputs, v, p
        widths = sum(w for _, w, _ in om.layers_of(kind))
        values = sum(int(np.prod(t)) for _, t in net._table.values()) + b * (widths + 1 + n_act)
        res = {"batch": b, "sources": len(net._hist_tags)}
        out["runs"].append(measure(net, x, y_r, a, (dx, dyr, da), args, res, 4 * values, values, host_alternative))
        del net
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--net", choices=("conv", "fork_vp", "discrate"), default="conv")
    ap.add_argument("--batch", type=int, default=None, help="conv: 1024; MLPs: 1024 and 65536")
    ap.add_argument("--calls", type=int, default=25)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    res = conv(args) if args.net == "conv" else mlp(args)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
