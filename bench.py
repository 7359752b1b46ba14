#!/usr/bin/env python
"""bench.py -- GA3C hot-path throughput on B200: TPS (training frames/s) and PPS (predictions/s).

    python bench.py --gpus N --steps K --warmup W            our arm (CUDA path through the C-ABI)
    python bench.py --impl reference --gpus N --steps K ...  the reference arm: CPU restatement of the
                                                             reference TF graph on the host cores

Workload (BASELINE.json configs[2] / configs[1], SURVEY.md 8d): conv NetworkVP, 84x84x4 fp32 frames,
6 actions.  A "step" is one batched A3C train step (forward, fused loss fwd/bwd, backward, gradient
allreduce when N>1, RMSProp) over B=1024 frames PER GPU (weak scaling).  `value` is the whole-job
training frames/s with inputs resident in HBM; `e2e` is the same step through Network.train() on
pinned HOST numpy buffers (H2D of the batch and D2H of the loss inside the timed region).  The `pps`
object is the ThreadPredictor path (Network.predict_p_and_v) at B=4096, measured the same two ways.

One JSON line on stdout (rank 0).  Everything else goes to stderr.

--dump-outputs DIR writes what the timed paths computed in their last step as DIR/<name>.npy (float32): the weights after
the last timed train step (train_<variable>.npy) and p / v of the last timed predict call (predict_p.npy, predict_v.npy).
The inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

STATE_DIM = 84 * 84 * 4
NUM_ACTIONS = 6
N_PARAMS = 1005623
L2_BYTES = 126 * 2 ** 20
_REAL_STDOUT = sys.stdout


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=float(d["hbm_gbs"]), tensor_burst=float(d["bf16_tflops"]),
                    tensor_sustained=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), source="measured")
    return dict(hbm=6650.0, tensor_burst=1590.0, tensor_sustained=1400.0, source="fallback")


def workload_config(args, world):
    return {"workload": f"NetworkVP 84x84x4 (conv8x8s4/16 -> conv4x4s2/32 -> fc256 -> 6 policy + 1 value), "
                        f"A3C train step B={args.batch}/GPU (BASELINE configs[2]); pps: predict B={args.predict_batch} "
                        f"(configs[1])",
            "train_batch_per_gpu": args.batch, "global_batch": args.batch * world, "predict_batch": args.predict_batch,
            "num_actions": NUM_ACTIONS, "frame": "84x84x4 fp32", "parallelism": f"dp{world}",
            "l2": "ring of device input batches > 126 MB L2, rotated every step"}


METRIC = "TPS: A3C training frames/s, NetworkVP 84x84x4 (PPS: predictions/s, in 'pps')"


# ------------------------------------------------------------------------------------------------
# algorithmic work per launch (DESIGN.md "Kernels"; SURVEY.md 8d).  bytes for HBM-bound kernels,
# flops for the tensor-bound dense1 GEMMs.
def kernel_work(name, b, train):
    n1, n2, fc = 441 * 16, 3872, 256
    x = STATE_DIM * 4
    xb = STATE_DIM * 2            # the bf16 copy of the frame conv_fwd leaves for the conv backward (live bytes; stored padded)
    if name == "conv_fwd":
        return "hbm", b * (x + (n1 * 2 + xb if train else 0) + n2 * 2)
    if name == "conv11_wgrad":
        return "hbm", b * (x + n1 * 2)
    if name == "conv12_bwd":      # split predecessor (GA3C_SPLIT_CONV_BWD)
        return "hbm", b * (n1 * 2 + n2 * 2 + n1 * 2)
    if name == "conv_bwd":        # fused conv12 dgrad + conv12 wgrad + conv11 wgrad: bf16 frame copy, n1, dn2 read once, dn1 stays on chip
        return "hbm", b * (xb + n1 * 2 + n2 * 2)
    if name == "heads":
        return "hbm", b * (fc * 4 + (fc * 2 + 4 + NUM_ACTIONS * 4 if train else (NUM_ACTIONS + 1) * 4))
    if name == "rmsprop":
        return "hbm", N_PARAMS * 20 + n2 * fc * 2
    if name == "dp_done":
        return "hbm", 128
    if name == "grad_reduce":     # L2-resident slabs: one slab per SM read, the small-tensor gradients written
        return "hbm", (148 + 1) * 14_500 * 4
    if name in ("dense_fwd", "dense_wgrad", "dense_dgrad"):
        return "tensor", 2.0 * b * n2 * fc
    if name == "dense_bwd":       # dgrad + wgrad tiles in one grid (dgrad alone in dp_mode='nccl')
        return "tensor", 4.0 * b * n2 * fc
    raise KeyError(name)


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clock and throttle reasons while the timed regions run (NVML, 50 ms period)."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._th = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception as e:      # noqa
            log(f"[bench] NVML unavailable: {e}")
            self._nv = None

    def _once(self):
        nv = self._nv
        self.samples.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
        r = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
            else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
        for name, bit in (("sw_power_cap", 0x4), ("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20),
                          ("hw_thermal_slowdown", 0x40), ("hw_power_brake", 0x80)):
            if r & bit:
                self.reasons.add(name)

    def start(self):
        if self._nv is None:
            return
        def loop():
            while not self._stop.is_set():
                try:
                    self._once()
                except Exception:   # noqa
                    pass
                self._stop.wait(0.05)
        self._th = threading.Thread(target=loop, daemon=True)
        self._th.start()

    def stop(self):
        if self._th is not None:
            self._stop.set()
            self._th.join()
            try:
                self._once()
            except Exception:       # noqa
                pass

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------
def synth_batch(rng, b):
    """Frames exactly as Environment.py:57-61 yields them (uint8 k -> k/128 - 1), returns U(-1,1),
    one-hot actions (SURVEY.md 8d)."""
    k = rng.integers(0, 256, size=(b, STATE_DIM), dtype=np.uint8)
    x = k.astype(np.float32)
    x *= np.float32(1 / 128.0)
    x -= np.float32(1.0)
    y_r = rng.uniform(-1.0, 1.0, size=b).astype(np.float32)
    a = np.eye(NUM_ACTIONS, dtype=np.float32)[rng.integers(0, NUM_ACTIONS, size=b)]
    return x, y_r, a


def cpu_reference_run(args, steps, warmup, budget_s=150.0):
    """The reference arm / cpu_baseline leg: torch-CPU fp32 restatement of the reference TF graph
    (oracle/oracle_torch.py; TensorFlow is not installable here), all host threads."""
    import torch
    from oracle import oracle_np as onp
    from oracle.oracle_torch import TorchNetworkVP
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    rng = np.random.default_rng(12345)
    net = TorchNetworkVP(onp.init_params(rng, NUM_ACTIONS))
    x, y_r, a = synth_batch(rng, args.batch)
    tx, tyr, ta = torch.from_numpy(x), torch.from_numpy(y_r), torch.from_numpy(a)
    # probe one step on 64 rows to size the bounded sample
    t0 = time.perf_counter()
    net.train(tx[:64], tyr[:64], ta[:64], 3e-4, 0.01)
    probe = time.perf_counter() - t0
    net.train(tx[:64], tyr[:64], ta[:64], 3e-4, 0.01)
    t0 = time.perf_counter()
    net.train(tx[:64], tyr[:64], ta[:64], 3e-4, 0.01)
    probe = min(probe, time.perf_counter() - t0)
    rows = args.batch
    while rows > 64 and probe * (rows / 64) * (steps + warmup) > budget_s:
        rows //= 2
    for _ in range(warmup):
        net.train(tx[:rows], tyr[:rows], ta[:rows], 3e-4, 0.01)
    t0 = time.perf_counter()
    for _ in range(steps):
        net.train(tx[:rows], tyr[:rows], ta[:rows], 3e-4, 0.01)
    dt = time.perf_counter() - t0
    tps = rows * steps / dt
    # predict leg
    prow = min(args.predict_batch, max(64, rows * 2))
    px = torch.from_numpy(synth_batch(rng, prow)[0])
    net.predict_p_and_v(px)
    psteps = max(2, min(steps, 10))
    t0 = time.perf_counter()
    for _ in range(psteps):
        net.predict_p_and_v(px)
    pdt = time.perf_counter() - t0
    return dict(tps=tps, ms_per_step=dt / steps * 1e3, rows=rows, steps=steps, cores=cores,
                pps=prow * psteps / pdt, prow=prow, psteps=psteps)


def run_reference(args, rank, world):
    if rank != 0:
        return
    r = cpu_reference_run(args, args.steps, args.warmup)
    sample = (f"{r['steps']} train steps of {r['rows']} frames (of B={args.batch}); "
              f"{r['psteps']} predict calls of {r['prow']} frames")
    out = {"impl": "reference", "metric": METRIC, "value": r["tps"], "unit": "frames/s", "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": workload_config(args, world),
           "cpu_baseline": {"value": r["tps"], "unit": "frames/s", "cores": r["cores"], "kind": "port", "sample": sample,
                            "note": "torch-CPU fp32 restatement of the reference TF graph (TensorFlow not installable)"},
           "e2e": {"value": r["tps"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "pps": {"value": r["pps"], "unit": "predictions/s", "batch": r["prow"]},
           "gpu_launches": 0}
    print(json.dumps(out), file=_REAL_STDOUT, flush=True)


# ------------------------------------------------------------------------------------------------
def mlp_flops(kind, s, a, train):
    """Algorithmic flops per sample of the config-4 MLPs: 2 per MAC; training = forward + weight gradients of every layer +
    data gradients of every layer but the first."""
    widths = [s, 4, 256, 256, 100, 64] if kind == "fork_vp" else [s, 10]
    n_out = 1 + 2 * a if kind == "fork_vp" else 1 + a
    macs = [widths[i] * widths[i + 1] for i in range(len(widths) - 1)] + [widths[-1] * n_out]
    fwd = 2.0 * sum(macs)
    return fwd * 3 - 2.0 * macs[0] if train else fwd


def run_mlp_section(args, dev, stream, pk, clocks):
    """BASELINE configs[3]: the fork's low-dimensional networks (fork NetworkVP S=3 A=1, NetworkVP_discrate S=4 A=2) at
    B = 1024 and 65,536, device-resident and end to end through the plugin API; fp32 SIMT kernels (ga3c_mlp_*)."""
    import torch
    from ga3c_b200 import mlp_network
    from oracle import oracle_mlp as om
    out = {"note": "BASELINE configs[3] (SURVEY 8a A6/A7): fp32 throughout; mlp_fused keeps a 64-row tile's activations in shared "
                   "memory through forward, heads, loss and the data-gradient chain; bound = fp32 FMA issue, not HBM"}
    sm_mhz = clocks.get("sm_max_mhz") or 1965
    fp32_peak = 148 * 128 * 2 * sm_mhz * 1e6 / 1e12          # TFLOP/s: 128 FMA lanes per SM per clock
    for kind, s, a, cls in (("fork_vp", 3, 1, mlp_network.NetworkVP), ("discrate", 4, 2, mlp_network.NetworkVP_discrate)):
        for b in (1024, 65536):
            rng = np.random.default_rng(12345)
            net = cls(f"gpu:{dev.index}", "bench_" + kind, a, s, max_batch=b, seed=12345)
            x = rng.uniform(-1, 1, size=(b, s)).astype(np.float32)
            y_r = rng.uniform(-1, 1, size=b).astype(np.float32)
            act = (rng.uniform(-1, 1, size=(b, a)).astype(np.float32) if kind == "fork_vp"
                   else np.eye(a, dtype=np.float32)[rng.integers(0, a, size=b)])
            dx, dyr, da = (torch.from_numpy(t).to(dev) for t in (x, y_r, act))
            p_out = torch.empty((b, a), dtype=torch.float32, device=dev)
            v_out = torch.empty((b,), dtype=torch.float32, device=dev)
            steps = args.steps

            def timed(fn):
                for _ in range(3):
                    fn()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                e0.record(stream)
                for _ in range(steps):
                    fn()
                e1.record(stream)
                torch.cuda.synchronize()
                return e0.elapsed_time(e1) / steps

            ms_t = timed(lambda: net.train_device(dx, dyr, da, stream=stream))
            ms_p = timed(lambda: net.predict_device(dx, p_out, v_out, stream=stream))
            net.kernel_timing(steps * 4)
            timed(lambda: net.train_device(dx, dyr, da, stream=stream))
            kt = {k: round(t / c * 1e3, 2) for k, (t, c) in net.kernel_times().items()}
            net.kernel_timing(0)
            t0 = time.perf_counter()
            for _ in range(steps):
                net.train(x, y_r, act, None, None, 0, fetch_losses=True)
            s_e2e_t = (time.perf_counter() - t0) / steps
            t0 = time.perf_counter()
            for _ in range(steps):
                net.predict_p_and_v(x)
            s_e2e_p = (time.perf_counter() - t0) / steps
            row = {"train_samples_per_s": b / (ms_t / 1e3), "train_ms": round(ms_t, 4),
                   "predictions_per_s": b / (ms_p / 1e3), "predict_ms": round(ms_p, 4),
                   "e2e_train_samples_per_s": b / s_e2e_t, "e2e_predictions_per_s": b / s_e2e_p,
                   "kernel_us": kt,
                   "fp32_tflops_train": round(mlp_flops(kind, s, a, True) * b / (ms_t / 1e3) / 1e12, 3),
                   "fp32_tflops_predict": round(mlp_flops(kind, s, a, False) * b / (ms_p / 1e3) / 1e12, 3),
                   "fp32_simt_peak_tflops": round(fp32_peak, 1)}
            if b == 65536:          # CPU port of the same step (numpy fp32 restatement, bounded sample)
                params = om.init_params(np.random.default_rng(1), kind, s, a)
                rows = 8192
                t0 = time.perf_counter()
                om.loss_and_grads(params, x[:rows], y_r[:rows], act[:rows], kind, dtype=np.float32)
                row["cpu_port_train_samples_per_s"] = rows / (time.perf_counter() - t0)
                row["cpu_port_sample"] = f"1 forward+backward of {rows} rows, numpy fp32 (oracle/oracle_mlp.py), {os.cpu_count()} cores visible"
            out[f"{kind}_S{s}_A{a}_B{b}"] = row
            del net
    return out


# ------------------------------------------------------------------------------------------------
DP_TOL = dict(max_abs=2e-4, rel_l2_of_update=0.15, entries_beyond_1e5=1000)


def oracle_distance(got, ref, start):
    """Distance of the weights after the data-parallel steps (`got`) from the oracle's (`ref`), both started at `start`.

    What the numbers look like (64 rows per rank, 2 steps, dp_check's seeded data):
      * a correct exchange differs from the oracle only where a stored bf16 activation, or a dense1 output next to zero (its
        ReLU gate), rounds the other way than in the fp64-accumulating oracle.  ONE such flip moves one entry of dense1/b by
        lr * dd1 and, through that row's dn2, a handful of conv weights: max |error| 2.8e-5 / 16 entries beyond 1e-5 / 0.025
        of the length of the update at world = 4; 1.6e-5 / 1 / 0.006 at world = 8; no flip at world = 2 (3e-8 / 0 / 6e-5).
        It does not scale with anything -- a batch has such a row or it has not (tools/dp_check_proxy.py reproduces the
        N-rank figures on one GPU to the last digit);
      * a broken exchange (a rank's rows missing from the sum, or counted twice; simulated with the oracle): max |error| 1.0e-3 to
        1.7e-3, 89 k to 158 k entries beyond 1e-5, error = 0.50 to 0.73 of the length of the update itself.
    The limits sit between the two with a factor >= 3 on either side: max |error| <= 2e-4, at most 1000 entries beyond 1e-5,
    and ||got - ref|| <= 0.15 ||ref - start||."""
    num = sum(float(((got[k].astype(np.float64) - ref[k]) ** 2).sum()) for k in got)
    den = sum(float(((ref[k].astype(np.float64) - start[k]) ** 2).sum()) for k in got)
    per = {k: float(np.abs(got[k] - ref[k]).max()) for k in got}
    worst = max(per.values())
    beyond = sum(int((np.abs(got[k] - ref[k]) > 1e-5).sum()) for k in got)
    rel = (num / max(den, 1e-300)) ** 0.5
    ok = worst <= DP_TOL["max_abs"] and rel <= DP_TOL["rel_l2_of_update"] and beyond <= DP_TOL["entries_beyond_1e5"]
    return dict(max_abs_vs_oracle=worst, worst_tensor=max(per, key=per.get), rel_l2_of_update=rel, entries_beyond_1e5=beyond,
                tol=dict(DP_TOL), ok=bool(ok))


def dp_check(net, rank, local_rank, world, B):
    """N > 1, before (and outside) the timed region: correctness of the data-parallel step at the benchmarked shape.
      1. the replicas start identical although no seed was given (rank 0's weights are broadcast at construction);
      2. two lock-step train steps at B rows per rank on rank-specific data leave bit-identical replicas (small tensors, their
         RMSProp slots, and the bf16 shadow of dense1/w that every rank holds);
      3. two steps at 64 rows per rank from the oracle's weights equal the oracle's two steps on the CONCATENATED batch (what a
         single ThreadTrainer fed all the rows would compute, SURVEY 8e).  The oracle is the checker here, nothing it does is timed.
    Any failure ends the run with a non-zero exit code."""
    import torch
    import torch.distributed as dist
    from oracle import oracle_np as onp
    dev = torch.device("cuda", local_rank)

    def replicas_identical():
        w = net.get_variables()
        ms, _ = net.get_slots()
        small = np.concatenate([w[k].ravel() for k in sorted(w) if k != "dense1/w:0"] +
                               [ms[k].ravel() for k in sorted(ms) if k != "dense1/w:0"])
        ok = True
        for arr in (small, net.workspace(6)):
            t = torch.from_numpy(np.ascontiguousarray(arr)).to(dev)
            got = [torch.empty_like(t) for _ in range(world)]
            dist.all_gather(got, t)
            ok = ok and all(torch.equal(got[0], g) for g in got)
        return ok

    rep = {"world": world}
    rep["identical_at_start_without_seed"] = replicas_identical()
    rng = np.random.default_rng(777 + rank)
    for _ in range(2):
        x, y_r, a = synth_batch(rng, B)
        net.train(x, y_r, a, None, None, 0)
    rep["replicas_identical"] = replicas_identical()
    rep["rows_per_rank"] = B
    # oracle leg
    rows = 64
    g = np.random.default_rng(4242)
    params = onp.init_params(g, NUM_ACTIONS)
    net.set_variables(params)
    net.set_slots({k: np.ones_like(v) for k, v in params.items()}, {k: np.zeros_like(v) for k, v in params.items()})
    ms, mom = onp.rmsprop_init(params)
    ref = params
    for _ in range(2):
        x = onp.synth_frames(g, rows * world)
        y_r, a = onp.synth_targets(g, rows * world, NUM_ACTIONS)
        net.train(x[rank * rows:(rank + 1) * rows], y_r[rank * rows:(rank + 1) * rows], a[rank * rows:(rank + 1) * rows], None, None, 0)
        if rank == 0:
            _, _, ref, ms, mom = onp.train_step(ref, ms, mom, x, y_r, a, lr=net.learning_rate, beta=net.beta, quant="bf16")
            ref = {k: v.astype(np.float32) for k, v in ref.items()}
    got = net.get_variables()
    dist_rep = oracle_distance(got, ref, params) if rank == 0 else dict(max_abs_vs_oracle=0.0, ok=True)
    rep["replicas_identical_oracle_leg"] = replicas_identical()
    rep.update(dist_rep, oracle_rows_per_rank=rows, oracle_steps=2,
               oracle="oracle_np.train_step (quant='bf16') on the concatenated batch")
    net.dp_check()
    ok = rep["identical_at_start_without_seed"] and rep["replicas_identical"] and rep["replicas_identical_oracle_leg"] and dist_rep["ok"]
    flag = torch.tensor([0 if ok else 1], device=dev)
    dist.all_reduce(flag)
    rep["ok"] = bool(flag.item() == 0)
    log(f"[bench] rank {rank} dp_check: {rep}")
    if not rep["ok"]:
        raise SystemExit(f"bench.py: data-parallel check FAILED on rank {rank}: {rep}")
    return rep


def dump_outputs(out_dir, variables, p_dev, v_dev):
    """--dump-outputs: 4 MB of weights plus 28 bytes per predicted row, below 64 MB for any predict batch that fits in HBM."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"train_" + k.replace(":0", "").replace("/", "_"): v for k, v in variables.items()}
    arrays.update(predict_p=p_dev.cpu().numpy(), predict_v=v_dev.cpu().numpy())
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float32))
    log(f"[bench] wrote {len(arrays)} arrays ({sum(a.nbytes for a in arrays.values()) / 2 ** 20:.1f} MB) to {out_dir}")


def run_ours(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    import ga3c_b200

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU fallback; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local_rank])

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    B, PB = args.batch, args.predict_batch
    K, W = args.steps, max(args.warmup, 3)
    numa = None
    if world > 1 and os.environ.get("GA3C_NUMA_BIND", "1") != "0":
        # threads (and the pinned buffers they first touch) next to this rank's GPU; N = 1 keeps every core for the CPU legs
        from ga3c_b200.numa import bind_to_gpu
        numa = bind_to_gpu(local_rank)
        log(f"[bench] rank {rank} numa: {numa}")
    # N > 1: no seed, as the reference constructor has none -- every rank draws its own weights and Network makes the
    # replicas equal rank 0's before the first step (checked below)
    net = ga3c_b200.Network(f"gpu:{local_rank}", "bench", NUM_ACTIONS, max_batch=max(B, PB), seed=12345 if world == 1 else None)
    pk = peaks()
    stream = torch.cuda.current_stream(dev)
    dp_report = dp_check(net, rank, local_rank, world, B) if world > 1 else None

    # ---- synthetic data: pinned host batches (e2e) and a device ring larger than L2 (value) ----
    rng = np.random.default_rng(12345 + 1000 * rank)
    n_ring = max(2, -(-int(1.5 * L2_BYTES) // (B * STATE_DIM * 4)) + 1)
    host = []
    for _ in range(min(n_ring, 2)):
        x, y_r, a = synth_batch(rng, B)
        host.append(tuple(torch.from_numpy(t).pin_memory() for t in (x, y_r, a)))
    ring = []
    for i in range(n_ring):
        hx, hyr, ha = host[i % len(host)]
        dx = hx.to(dev)
        if i >= len(host):                  # distinct contents per ring slot without more host RNG time
            dx = torch.roll(dx, shifts=i, dims=0)
        ring.append((dx, hyr.to(dev), ha.to(dev)))
    px_host = torch.from_numpy(synth_batch(rng, PB)[0]).pin_memory()
    n_pring = max(2, -(-int(1.5 * L2_BYTES) // (PB * STATE_DIM * 4)) + 1)
    pring = [torch.roll(px_host.to(dev), shifts=i, dims=0) for i in range(n_pring)]
    p_out = torch.empty((PB, NUM_ACTIONS), dtype=torch.float32, device=dev)
    v_out = torch.empty((PB,), dtype=torch.float32, device=dev)
    torch.cuda.synchronize()

    def timed(fn, steps):
        """barrier + sync on both sides, CUDA events on the launching stream, max over ranks (ms)."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier(); torch.cuda.synchronize()
        e0.record(stream)
        for i in range(steps):
            fn(i)
        e1.record(stream)
        torch.cuda.synchronize(); barrier()
        return max_over_ranks(e0.elapsed_time(e1))

    def train_step(i):
        dx, dyr, da = ring[i % n_ring]
        net.train_device(dx, dyr, da, stream=stream)

    def predict_step(i):
        net.predict_device(pring[i % n_pring], p_out, v_out, stream=stream)

    sampler = ClockSampler(local_rank)
    for i in range(W):
        train_step(i)
    for i in range(W):
        predict_step(i)
    torch.cuda.synchronize()

    sampler.start()
    l0 = net.launch_count()
    ms_train = timed(train_step, K)
    launches = net.launch_count() - l0
    ms_pred = timed(predict_step, K)
    if args.dump_outputs and rank == 0:         # before the legs below train further
        dump_outputs(args.dump_outputs, net.get_variables(), p_out, v_out)

    # spread: the same K steps timed in blocks of <= 10 (SURVEY 8d asks for median and best next to the mean)
    blocks = []
    done = 0
    while done < K:
        nb = min(10, K - done)
        blocks.append(timed(lambda i, d=done: train_step(d + i), nb) / nb)
        done += nb

    # ---- per-kernel durations, live, with events on the launch stream (roofline leg) ----
    net.kernel_timing(K * 10)
    ms_train_ev = timed(train_step, K)
    kt_train = net.kernel_times()
    net.kernel_timing(K * 3)
    ms_pred_ev = timed(predict_step, K)
    kt_pred = net.kernel_times()
    net.kernel_timing(0)
    # the same step seen WITHOUT serialising the programmatic-dependent-launch chain: globaltimer stamps per kernel
    # (first CTA past its dependency wait -> last CTA ended), one traced step each
    torch.cuda.synchronize()
    net.trace_begin(stream)
    train_step(0)
    tr_train = {k: round(v[5] - v[2], 2) for k, v in net.trace_end().items()}
    net.trace_begin(stream)
    predict_step(0)
    tr_pred = {k: round(v[5] - v[2], 2) for k, v in net.trace_end().items()}
    log(f"[bench] rank {rank} train kernels (us): " + ", ".join(f"{k} {t / max(c, 1) * 1e3:.1f}" for k, (t, c) in kt_train.items() if c))

    # ---- e2e through the public API on pinned host buffers ----
    def e2e(fn, steps):
        barrier(); torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(steps):
            fn(i)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        barrier()
        return max_over_ranks(dt)

    def train_e2e(i):
        hx, hyr, ha = host[i % len(host)]
        net.train(hx.numpy(), hyr.numpy(), ha.numpy(), None, None, 0, fetch_losses=True)

    def predict_e2e(i):
        net.predict_p_and_v(px_host.numpy())

    # the reference's configuration: Config.TRAINERS = 2 ThreadTrainers call Network.train concurrently (Config.py:59,
    # ThreadTrainer.py:42-62); the copy of one call overlaps the kernels and the wake-up of the other
    def e2e_threads(fn, steps, nthreads=2):
        import threading
        barrier(); torch.cuda.synchronize()
        errs = []

        def work(t):
            try:
                for i in range(t, steps, nthreads):
                    fn(i, t)
            except Exception as ex:          # noqa
                errs.append(ex)
        ths = [threading.Thread(target=work, args=(t,)) for t in range(nthreads)]
        t0 = time.perf_counter()
        for th in ths:
            th.start()
        for th in ths:
            th.join()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        barrier()
        if errs:
            raise errs[0]
        return max_over_ranks(dt)

    def train_e2e_t(i, t):
        hx, hyr, ha = host[i % len(host)]
        net.train(hx.numpy(), hyr.numpy(), ha.numpy(), None, None, t, fetch_losses=True)

    k_e2e = K
    for i in range(2):
        train_e2e(i); predict_e2e(i); train_e2e_t(i, 1)
    s_train_e2e = e2e(train_e2e, k_e2e)
    # data parallel: every rank must enter every exchange step in the same order -- two free-running trainer threads per rank
    # would not; the lock-step trainer is single-threaded there
    s_train_e2e_2t = e2e_threads(train_e2e_t, k_e2e) if world == 1 else None
    s_pred_e2e = e2e(predict_e2e, k_e2e)

    # the drop-in case: the reference's ThreadTrainer hands over PAGEABLE arrays (np.concatenate output, ThreadTrainer.py:54-58)
    pageable = [tuple(np.array(t.numpy(), copy=True) for t in h) for h in host]

    def train_e2e_pageable(i):
        x, y_r, a = pageable[i % len(pageable)]
        net.train(x, y_r, a, None, None, 0, fetch_losses=True)

    def train_e2e_pageable_t(i, t):
        x, y_r, a = pageable[i % len(pageable)]
        net.train(x, y_r, a, None, None, t, fetch_losses=True)

    train_e2e_pageable(0)
    s_train_e2e_pg = e2e(train_e2e_pageable, k_e2e)
    s_train_e2e_pg_2t = e2e_threads(train_e2e_pageable_t, k_e2e) if world == 1 else None
    # how the pageable array reaches the pinned staging buffer (Network._h2d): the library's worker threads with streaming
    # stores (ga3c_stage_h2d, the default), the same with plain stores, or torch's copy from the calling thread
    pg_variants = {}
    if world == 1:
        saved = {k: os.environ.get(k) for k in ("GA3C_COPY_THREADS", "GA3C_COPY_NT")}
        try:
            for name, threads, nt in (("torch_copy_from_the_caller", 0, 1), ("native_4_threads", 4, 1), ("native_8_threads", 8, 1),
                                      ("native_12_threads", 12, 1), ("native_8_threads_plain_stores", 8, 0)):
                os.environ["GA3C_COPY_THREADS"], os.environ["GA3C_COPY_NT"] = str(threads), str(nt)
                train_e2e_pageable(0)
                one = e2e(train_e2e_pageable, k_e2e)
                two = e2e_threads(train_e2e_pageable_t, k_e2e)
                pg_variants[name] = {"two_trainers": round(B * k_e2e / two), "single_caller": round(B * k_e2e / one)}
        finally:
            for k, v in saved.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v

    # the ceiling of any fp32-contract e2e number: a bare pinned host -> device copy of one batch, all ranks at once
    def h2d_only(i):
        hx, _, _ = host[i % len(host)]
        ring[i % n_ring][0].copy_(hx, non_blocking=True)

    h2d_only(0)
    s_h2d = e2e(h2d_only, k_e2e)
    h2d_ceiling_gbs = B * STATE_DIM * 4 * k_e2e / s_h2d / 1e9

    # ---- uint8 frame ingestion (SURVEY 8f F2), reported separately: a different input contract (raw pixels, x = k/128 - 1
    # applied on the GPU; outputs bit-identical to the fp32 path) with 4x fewer H2D and HBM input bytes ----
    hx8 = [(torch.clamp((h[0] + 1.0) * 128.0, 0, 255)).to(torch.uint8).pin_memory() for h in host]
    px8_host = (torch.clamp((px_host + 1.0) * 128.0, 0, 255)).to(torch.uint8).pin_memory()
    n_ring8 = max(2, -(-int(1.5 * L2_BYTES) // (B * STATE_DIM)) + 1)
    ring8 = [(torch.roll(hx8[i % len(hx8)].to(dev), shifts=i, dims=0), ring[i % n_ring][1], ring[i % n_ring][2]) for i in range(n_ring8)]
    n_pring8 = max(2, -(-int(1.5 * L2_BYTES) // (PB * STATE_DIM)) + 1)
    pring8 = [torch.roll(px8_host.to(dev), shifts=i, dims=0) for i in range(n_pring8)]

    def train_step8(i):
        dx, dyr, da = ring8[i % n_ring8]
        net.train_device(dx, dyr, da, stream=stream)

    def predict_step8(i):
        net.predict_device(pring8[i % n_pring8], p_out, v_out, stream=stream)

    def train_e2e8(i):
        _, hyr, ha = host[i % len(host)]
        net.train(hx8[i % len(hx8)].numpy(), hyr.numpy(), ha.numpy(), None, None, 0, fetch_losses=True)

    def predict_e2e8(i):
        net.predict_p_and_v(px8_host.numpy())

    for i in range(W):
        train_step8(i); predict_step8(i)
    torch.cuda.synchronize()
    ms_train8 = timed(train_step8, K)
    ms_pred8 = timed(predict_step8, K)
    for i in range(2):
        train_e2e8(i); predict_e2e8(i)
    s_train_e2e8 = e2e(train_e2e8, k_e2e)

    def train_e2e8_t(i, t):
        _, hyr, ha = host[i % len(host)]
        net.train(hx8[i % len(hx8)].numpy(), hyr.numpy(), ha.numpy(), None, None, t, fetch_losses=True)

    if world == 1:
        train_e2e8_t(1, 1)
    s_train_e2e8_2t = e2e_threads(train_e2e8_t, k_e2e) if world == 1 else None
    s_pred_e2e8 = e2e(predict_e2e8, k_e2e)
    sampler.stop()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    def roofline(kt, b, train, total_ms_events):
        rows = {}
        for name, (tot, cnt) in kt.items():
            if cnt == 0:
                continue
            bound, work = kernel_work(name, b, train)
            avg_s = tot / cnt / 1e3
            if bound == "hbm":
                ach, peak, unit = work / avg_s / 1e9, pk["hbm"], "GB/s"
            else:
                ach, peak, unit = work / avg_s / 1e12, pk["tensor_sustained"], "TFLOP/s"
            rows[name] = {"bound": bound, "achieved": round(ach, 1), "peak": peak, "unit": unit,
                          "frac": round(ach / peak, 4), "avg_us": round(avg_s * 1e6, 2),
                          "share": round(tot / total_ms_events, 4), "launches": int(cnt)}
        return rows

    rf_train = roofline(kt_train, B, True, ms_train_ev)
    rf_pred = roofline(kt_pred, PB, False, ms_pred_ev)
    top = max(rf_train, key=lambda k: rf_train[k]["share"])
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")      # dram bytes per launch from the committed ncu capture
    if os.path.exists(tpath):
        traffic = json.load(open(tpath)).get(top)
    in_step = None
    if tr_train.get(top):
        bound_t, work_t = kernel_work(top, B, True)
        peak_t = pk["hbm"] if bound_t == "hbm" else pk["tensor_sustained"]
        in_step = round(work_t / (tr_train[top] * 1e-6) / (1e9 if bound_t == "hbm" else 1e12) / peak_t, 4)
    roof = dict(rf_train[top], kernel=top, traffic=traffic, peak_source=pk["source"], frac_in_step=in_step,
                note="achieved = algorithmic bytes (or flops) per launch / CUDA-event duration of that kernel, "
                     "measured in this run on the launch stream",
                kernels_train=rf_train, kernels_predict=rf_pred,
                step_ms_with_events=round(ms_train_ev / K, 4),
                in_step_us={"note": "per-kernel busy time inside the pipelined step (ga3c_trace_*: first CTA started -> last CTA "
                                    "ended, one traced step); event brackets above serialise the launch chain and read 3-8 us longer",
                            "train": tr_train, "predict": tr_pred})

    tps = world * B * K / (ms_train / 1e3)
    pps = world * PB * K / (ms_pred / 1e3)
    s_e2e_head = s_train_e2e_2t if s_train_e2e_2t is not None else s_train_e2e
    out = {"metric": METRIC, "value": tps, "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": W,
           "ms_per_step": ms_train / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "bf16", "data": "synthetic", "config": workload_config(args, world),
           "tps_batches_per_s": tps / B,
           "ms_per_step_blocks": {"note": "the K steps again, in blocks of <= 10 (barrier + sync per block)", "n": len(blocks),
                                  "best": round(min(blocks), 5), "median": round(float(np.median(blocks)), 5)},
           "roofline": roof,
           "e2e": {"value": world * B * k_e2e / s_e2e_head, "unit": "frames/s",
                   "h2d_bytes_per_step": B * (STATE_DIM + 1 + NUM_ACTIONS) * 4, "d2h_bytes_per_step": 16,
                   "h2d_gbs_per_gpu": round(B * (STATE_DIM + 1 + NUM_ACTIONS) * 4 * k_e2e / s_e2e_head / 1e9, 2),
                   "steps": k_e2e, "trainer_threads": 2 if s_train_e2e_2t is not None else 1,
                   "api": ("Network.train(x, y_r, a, x2, done, trainer_id) on pinned host numpy, called by Config.TRAINERS = 2 trainer "
                           "threads as the reference's Server does (every call: H2D of its batch, the step, D2H of the losses, sync)")
                          if s_train_e2e_2t is not None else
                          "Network.train(x, y_r, a, x2, done, trainer_id) on pinned host numpy, one caller (lock-step data parallel)",
                   "single_caller": {"value": world * B * k_e2e / s_train_e2e, "unit": "frames/s",
                                     "note": "the same calls from ONE thread: nothing overlaps the copy of the next batch"},
                   "h2d_ceiling_gbs_per_gpu": round(h2d_ceiling_gbs, 2),
                   "frac_of_h2d_ceiling": round(B * (STATE_DIM + 1 + NUM_ACTIONS) * 4 * k_e2e / s_e2e_head / 1e9 / h2d_ceiling_gbs, 3),
                   "ceiling_note": "bare cudaMemcpyAsync of one pinned fp32 batch per step, all ranks at once, same box and run",
                   "pageable": {"value": world * B * k_e2e / (s_train_e2e_pg_2t or s_train_e2e_pg), "unit": "frames/s",
                                "single_caller": world * B * k_e2e / s_train_e2e_pg,
                                "api": "the same calls on ordinary (pageable) numpy arrays, what the reference's ThreadTrainer hands "
                                       "over (np.concatenate output): a chunked host copy into pinned staging (ga3c_stage_h2d: "
                                       "worker threads of the library, streaming stores) overlaps the DMA",
                                "copy_threads": ga3c_b200.Network._copy_threads(),
                                "variants_frames_per_s": pg_variants}},
           "pps": {"value": pps, "unit": "predictions/s", "batch": PB, "ms_per_step": ms_pred / K,
                   "e2e": {"value": world * PB * k_e2e / s_pred_e2e, "unit": "predictions/s",
                           "h2d_bytes_per_step": PB * STATE_DIM * 4, "d2h_bytes_per_step": PB * (NUM_ACTIONS + 1) * 4,
                           "api": "Network.predict_p_and_v(x) on pinned host numpy"}},
           "uint8_frames": {"note": "SURVEY 8f F2, a different input contract (raw uint8 pixels, k/128-1 applied in the kernels; "
                                    "outputs bit-identical to the fp32 path): not comparable with `value` / `e2e` byte for byte",
                            "value": world * B * K / (ms_train8 / 1e3), "unit": "frames/s", "ms_per_step": ms_train8 / K,
                            "e2e": {"value": world * B * k_e2e / (s_train_e2e8_2t or s_train_e2e8), "unit": "frames/s",
                                    "trainer_threads": 2 if s_train_e2e8_2t is not None else 1,
                                    "single_caller": world * B * k_e2e / s_train_e2e8,
                                    "h2d_bytes_per_step": B * (STATE_DIM + (1 + NUM_ACTIONS) * 4), "d2h_bytes_per_step": 16},
                            "pps": {"value": world * PB * K / (ms_pred8 / 1e3), "unit": "predictions/s", "ms_per_step": ms_pred8 / K,
                                    "e2e": {"value": world * PB * k_e2e / s_pred_e2e8, "unit": "predictions/s",
                                            "h2d_bytes_per_step": PB * STATE_DIM, "d2h_bytes_per_step": PB * (NUM_ACTIONS + 1) * 4}}},
           "gpu_launches": int(launches),
           "clocks": sampler.summary()}
    if dp_report is not None:
        out["dp_check"] = dp_report
    if numa is not None:
        out["numa"] = numa

    if world == 1 and not args.no_mlp:
        out["mlp"] = run_mlp_section(args, dev, stream, pk, out["clocks"])
    if world == 1 and not args.no_cpu_baseline:
        log("[bench] timing the CPU restatement (bounded sample) ...")
        r = cpu_reference_run(args, steps=args.cpu_steps, warmup=1, budget_s=25.0)
        out["cpu_baseline"] = {"value": r["tps"], "unit": "frames/s", "cores": r["cores"], "kind": "port",
                               "sample": f"{r['steps']} train steps of {r['rows']} frames (of B={B})",
                               "pps": r["pps"],
                               "note": "torch-CPU fp32 restatement of the reference TF graph (TensorFlow not installable)"}
    print(json.dumps(out), file=_REAL_STDOUT, flush=True)
    if world > 1:
        dist.destroy_process_group()


def _claim_stdout():
    """Library chatter (NCCL prints its version on stdout) must not pollute the one-JSON-line contract:
    point fd 1 at stderr for the whole run and keep the real stdout for the final line."""
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    return real


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=1024, help="train frames per GPU per step")
    ap.add_argument("--predict-batch", type=int, default=4096)
    ap.add_argument("--cpu-steps", type=int, default=10)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-mlp", action="store_true", help="skip the configs[3] low-dimensional MLP section")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed train and predict steps as "
                                                          "DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    global _REAL_STDOUT
    _REAL_STDOUT = _claim_stdout()
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
