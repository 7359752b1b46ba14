"""`Network` -- drop-in for the reference's Network plugin (NetworkVP.py:36-288) on the conv
NetworkVP (conv11 8x8s4/16 -> conv12 4x4s2/32 -> dense1 256 -> value + policy heads;
NetworkDNav.py:81-90 trunk, NetworkVP_discrate.py:60-130 heads/loss/optimizer).

Same constructor, attributes and methods as the reference class:
    Network(device, model_name, num_actions, state_dim)
    .learning_rate, .beta          mutable, read at every train() (NetworkVP.py:230-231; Server.py:174-175)
    predict_p_and_v(x) -> [p, v]   (NetworkVP.py:248-252)
    train(x, y_r, a, x2, done, trainer_id)   (NetworkVP.py:254-257)
    log / histograms / save / load / predict_single / predict_p / predict_v / get_global_step /
    get_variables_names / get_variable_value

PyTorch is used for pinned host staging, device buffers, streams and torch.distributed only; every
kernel is launched by the C-ABI library (include/ga3c_b200.h).  No CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os
import threading
import warnings

import numpy as np
import torch

from . import _capi, summaries
from ._arena import ArenaNetworkMixin, _parse_device  # noqa: F401  (_parse_device: part of this module's interface)
from .config import Config as _DefaultConfig

STATE_DIM = 84 * 84 * 4


def geometry(cfg):
    """(IMAGE_HEIGHT, IMAGE_WIDTH, STACKED_FRAMES) of a Config, 84 / 84 / 4 where it has no such attribute (Config.py:90-92).
    Raises ValueError naming the knob outside 1..256 / 1..256 / 1..8."""
    out = []
    for knob, default, hi in (("IMAGE_HEIGHT", 84, 256), ("IMAGE_WIDTH", 84, 256), ("STACKED_FRAMES", 4, 8)):
        v = int(getattr(cfg, knob, default))
        if not 1 <= v <= hi:
            raise ValueError(f"Config.{knob} must be 1..{hi}, got {v}")
        out.append(v)
    return tuple(out)


class _DevArray:
    """Exposes a raw device allocation owned by the C library through __cuda_array_interface__."""

    def __init__(self, ptr: int, n: int, owner):
        self._owner = owner
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f4", "data": (ptr, False), "version": 2}


class _HandleLock:
    """`with lock:` on the handle's own mutex (ga3c_lock / ga3c_unlock): shared with the native predictor batcher, which runs
    outside the interpreter.  ctypes releases the GIL while a thread waits for it."""

    def __init__(self, lib, handle):
        self._lib, self._h = lib, handle

    def __enter__(self):
        self._lib.ga3c_lock(self._h)
        return self

    def __exit__(self, *exc):
        self._lib.ga3c_unlock(self._h)
        return False


class _TrainSlot:
    """Staging of ONE trainer thread.  The reference runs Config.TRAINERS (= 2, Config.py:59) ThreadTrainers that call
    Network.train concurrently (ThreadTrainer.py:42-62, Server.py:141-150): call k+1's host -> device copy goes into the other
    slot, on that slot's own stream, while call k's kernels run and its caller waits for them -- PCIe never idles between
    steps.  Slot = trainer_id % 2; a slot is used by one call at a time (its lock)."""

    def __init__(self, tdev, state_dim):
        self.lock = threading.Lock()
        self.tdev = tdev
        self.state_dim = state_dim
        self.rows = 0
        self.rows8 = 0
        with torch.cuda.device(tdev):
            self.stream = torch.cuda.Stream(device=tdev)
            self.ready = torch.cuda.Event()

    def buffers(self, rows: int, num_actions: int, u8: bool):
        with torch.cuda.device(self.tdev):
            if rows > self.rows:
                self.hyr = torch.empty((rows,), dtype=torch.float32, pin_memory=True)
                self.ha = torch.empty((rows, num_actions), dtype=torch.float32, pin_memory=True)
                self.dyr = torch.empty((rows,), dtype=torch.float32, device=self.tdev)
                self.da = torch.empty((rows, num_actions), dtype=torch.float32, device=self.tdev)
                self.hx = torch.empty((rows, self.state_dim), dtype=torch.float32, pin_memory=True)
                self.dx = torch.empty((rows, self.state_dim), dtype=torch.float32, device=self.tdev)
                self.rows = rows
            if u8 and rows > self.rows8:
                self.hx8 = torch.empty((rows, self.state_dim), dtype=torch.uint8, pin_memory=True)
                self.dx8 = torch.empty((rows, self.state_dim), dtype=torch.uint8, device=self.tdev)
                self.rows8 = rows
        return (self.hx8, self.dx8) if u8 else (self.hx, self.dx)


class Network(ArenaNetworkMixin):
    def __init__(self, device, model_name, num_actions, state_dim=None, *, config=None, max_batch=None,
                 seed=None, data_parallel=None, dp_mode=None):
        """state_dim (default: the Config's H*W*C) must equal IMAGE_HEIGHT * IMAGE_WIDTH * STACKED_FRAMES of `config`."""
        cfg = config or _DefaultConfig
        if state_dim is None:
            state_dim = int(np.prod(geometry(cfg)))
        sd = int(np.prod(state_dim)) if not isinstance(state_dim, int) else state_dim
        h, w, nc = self.geometry = geometry(cfg)
        if sd != h * w * nc:
            raise ValueError(f"conv NetworkVP expects state_dim = IMAGE_HEIGHT*IMAGE_WIDTH*STACKED_FRAMES = {h}*{w}*{nc} = "
                             f"{h * w * nc}, got {sd}")
        fields = self._setup(device, model_name, num_actions, sd, cfg, max_batch)
        c = _capi.ga3c_config(device=self._ordinal, num_actions=self.num_actions, max_batch=self._max_batch,
                              image_height=h, image_width=w, stacked_frames=nc, **fields)
        h = C.c_void_p()
        _capi.check(self._lib.ga3c_create(C.byref(c), C.byref(h)), "ga3c_create")
        self._h = h
        self._lock = _HandleLock(self._lib, self._h)

        # name -> (offset, shape) table in TF creation order
        self._table = {}
        for i in range(self._lib.ga3c_param_count(self._h)):
            name, off, nd = C.c_char_p(), C.c_int64(), C.c_int32()
            shape = (C.c_int64 * 4)()
            _capi.check(self._lib.ga3c_param_info(self._h, i, C.byref(name), C.byref(off), C.byref(nd), shape),
                        "ga3c_param_info")
            self._table[name.value.decode()] = (off.value, tuple(shape[k] for k in range(nd.value)))
        self._arena_floats = self._lib.ga3c_arena_floats(self._h)
        ptrs = [C.c_void_p() for _ in range(4)]
        _capi.check(self._lib.ga3c_arena_ptrs(self._h, *[C.byref(p) for p in ptrs]), "ga3c_arena_ptrs")
        with torch.cuda.device(self._tdev):
            self._grad_arena = torch.as_tensor(_DevArray(ptrs[1].value, self._arena_floats, self), device=self._tdev)
            self._param_arena = torch.as_tensor(_DevArray(ptrs[0].value, self._arena_floats, self), device=self._tdev)
            self._stream = torch.cuda.Stream(device=self._tdev)
            self._loss_dev = torch.zeros(4, dtype=torch.float32, device=self._tdev)
        self._alloc_io(self._max_batch)
        self._train_slots = [_TrainSlot(self._tdev, self.state_dim) for _ in range(2)]     # staging per trainer thread, allocated on first use

        # variable init: U(-d, d), d = 1/sqrt(fan_in)  (NetworkVP.py:214-217, NetworkDNav.py:258-261)
        rng = np.random.default_rng(seed)
        fan_in = {"conv11": 8 * 8 * self.geometry[2], "conv12": 4 * 4 * 16, "dense1": self._table["dense1/w:0"][1][0],
                  "logits_v": 256, "logits_p": 256}
        init = {}
        for name, (_, shape) in self._table.items():
            d = 1.0 / np.sqrt(fan_in[name.split("/")[0]])
            init[name] = rng.uniform(-d, d, size=shape).astype(np.float32)
        self.set_variables(init)

        # data parallelism: gradients are SUM-allreduced (no averaging: the loss is sum-reduced,
        # NetworkVP_discrate.py:61,:83-85), then every rank applies the identical RMSProp update
        #   dp_mode "fused" (default): reduce-scatter + RMSProp + all-gather in ONE kernel over CUDA-IPC peer
        #                             memory (ga3c_dp_attach); no collective library call on the step's critical path
        #   dp_mode "nccl"          : two-segment NCCL allreduce overlapping the conv backward, then local RMSProp
        from .dataparallel import GradientAllReduce, exchange_ipc_handles
        self._allreduce = GradientAllReduce(self._grad_arena, self._table["dense1/w:0"][0])
        if data_parallel is False:
            self._allreduce.enabled = False
        self.dp_mode = None
        self._allreduce2 = None
        if self._allreduce.enabled:
            self.dp_mode = dp_mode or os.environ.get("GA3C_DP", "fused")
            if self.dp_mode not in ("fused", "nccl"):
                raise ValueError(f"dp_mode must be 'fused' or 'nccl', got {self.dp_mode!r}")
        if self.dp_mode == "fused" and (getattr(cfg, "USE_GRAD_CLIP", False) or self._dual or self.geometry != (84, 84, 4)):
            # the per-variable norms need the whole reduced gradient, and DUAL_RMSPROP has two gradient arenas: allreduce
            # first (NCCL), then clip / update locally; the peer-memory exchange is built around the 84x84x4 arena
            self.dp_mode = "nccl"
        if self._allreduce.enabled and self._dual:
            g2 = C.c_void_p()
            _capi.check(self._lib.ga3c_arena_ptr(self._h, 4, C.byref(g2)), "ga3c_arena_ptr")
            with torch.cuda.device(self._tdev):
                self._grad2_arena = torch.as_tensor(_DevArray(g2.value, self._arena_floats, self), device=self._tdev)
            self._allreduce2 = GradientAllReduce(self._grad2_arena, self._table["dense1/w:0"][0])
        if self._allreduce.enabled:
            # Replicas must START identical: the reference constructor has no seed argument (NetworkVP.py:37), so every rank
            # drew its own U(+-1/sqrt(fan_in)) weights above.  Rank 0's weights and slots win.
            self.sync_replicas()
        if self.dp_mode == "fused":
            import torch.distributed as dist
            n = self._lib.ga3c_dp_handle_bytes()
            mine = C.create_string_buffer(n)
            _capi.check(self._lib.ga3c_dp_export(self._h, mine), "ga3c_dp_export")
            handles = exchange_ipc_handles(mine.raw, self._tdev)
            _capi.check(self._lib.ga3c_dp_attach(self._h, dist.get_rank(), dist.get_world_size(), handles),
                        "ga3c_dp_attach")
            dist.barrier(device_ids=[self._ordinal])      # every rank has mapped every slab before the first step
        self._dp = self.dp_mode == "nccl"
        self._hist_tags = summaries.histogram_tags(self._table)

    # ------------------------------------------------------------------ buffers
    def _alloc_io(self, rows: int):
        super()._alloc_io(rows)
        self._hx8 = self._dx8 = None          # uint8 frame staging, allocated on first use (F2 ingestion)

    def _io_u8(self):
        if self._hx8 is None or self._hx8.shape[0] < self._io_rows:
            with torch.cuda.device(self._tdev):
                self._hx8 = torch.empty((self._io_rows, self.state_dim), dtype=torch.uint8, pin_memory=True)
                self._dx8 = torch.empty((self._io_rows, self.state_dim), dtype=torch.uint8, device=self._tdev)
        return self._hx8, self._dx8

    @staticmethod
    def _frames(x, state_dim):
        """Frames as handed over: float32 [B, state_dim] (the reference contract), or uint8 [B, state_dim] raw pixels
        (F2 ingestion: x = k/128 - 1, Environment.py:60, is applied on the GPU; outputs are bit-identical)."""
        x = np.asarray(x)
        if x.dtype != np.uint8:
            x = np.asarray(x, dtype=np.float32)
        if x.ndim != 2 or x.shape[1] != state_dim:
            x = x.reshape(x.shape[0], -1)
            if x.shape[1] != state_dim:
                raise ValueError(f"x must be [B, {state_dim}], got {x.shape}")
        return x

    _CHUNK_BYTES = 8 << 20

    @staticmethod
    def _copy_threads() -> int:
        """Worker threads of ga3c_stage_h2d for one pageable array: GA3C_COPY_THREADS, else half of this rank's share of the
        cores this process may run on, between 2 and 8 (0: the interpreter-side chunked copy)."""
        env = os.environ.get("GA3C_COPY_THREADS")
        if env is not None:
            return max(0, int(env))
        cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 2)
        ranks = max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))
        return max(2, min(8, cores // (2 * ranks)))

    def _h2d(self, arr: np.ndarray, pinned: torch.Tensor, dst: torch.Tensor, b: int):
        """Enqueues the host -> device copy of arr[:b] on the current stream.  A pinned caller array is copied as it is; a
        pageable one (what the reference's ThreadTrainer hands over: np.concatenate output, ThreadTrainer.py:54-58) goes
        through this Network's pinned staging buffer in chunks, so that the host copy of chunk k+1 overlaps the DMA of chunk k
        instead of preceding the whole transfer: by the library's worker threads with streaming stores (ga3c_stage_h2d, no
        interpreter involved), or with GA3C_COPY_THREADS=0 by torch's copy from this thread."""
        src = None
        if arr.flags["C_CONTIGUOUS"] and arr.flags["WRITEABLE"]:
            src = torch.from_numpy(arr)
            if src.is_pinned():
                dst[:b].copy_(src, non_blocking=True)
                return
        if arr.nbytes <= self._CHUNK_BYTES or not arr.flags["C_CONTIGUOUS"]:
            pinned[:b].numpy()[...] = arr
            dst[:b].copy_(pinned[:b], non_blocking=True)
            return
        threads = self._copy_threads()
        if threads > 0:
            st = torch.cuda.current_stream(self._tdev)
            _capi.check(self._lib.ga3c_stage_h2d(dst.data_ptr(), pinned.data_ptr(), arr.ctypes.data, arr[:b].nbytes,
                                                 self._CHUNK_BYTES, threads, st.cuda_stream), "ga3c_stage_h2d")
            return
        if src is None:
            pinned[:b].numpy()[...] = arr
            dst[:b].copy_(pinned[:b], non_blocking=True)
            return
        rows = max(1, self._CHUNK_BYTES // max(1, arr[0].nbytes))
        for lo in range(0, b, rows):
            hi = min(b, lo + rows)
            pinned[lo:hi].copy_(src[lo:hi])
            dst[lo:hi].copy_(pinned[lo:hi], non_blocking=True)

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                self._lib.ga3c_dp_detach(self._h)
        except Exception:
            pass
        super().__del__()

    # ------------------------------------------------------------------ device-resident API
    def predict_device(self, x_dev: torch.Tensor, p_out: torch.Tensor = None, v_out: torch.Tensor = None, stream=None):
        """predict_p_and_v on tensors already in HBM.  Asynchronous on `stream` (default: current)."""
        b = x_dev.shape[0]
        self._ensure(b)
        if p_out is None:
            p_out = torch.empty((b, self.num_actions), dtype=torch.float32, device=self._tdev)
        if v_out is None:
            v_out = torch.empty((b,), dtype=torch.float32, device=self._tdev)
        st = stream or torch.cuda.current_stream(self._tdev)
        fn = self._lib.ga3c_predict_u8 if x_dev.dtype == torch.uint8 else self._lib.ga3c_predict
        _capi.check(fn(self._h, x_dev.data_ptr(), b, p_out.data_ptr(), v_out.data_ptr(), st.cuda_stream), "ga3c_predict")
        return p_out, v_out

    def train_device(self, x_dev, yr_dev, a_dev, *, loss_out: torch.Tensor = None, stream=None):
        """One A3C step on tensors already in HBM (forward, loss fwd/bwd, backward, [allreduce], RMSProp)."""
        b = x_dev.shape[0]
        self._ensure(b)
        st = stream or torch.cuda.current_stream(self._tdev)
        loss_ptr = loss_out.data_ptr() if loss_out is not None else None
        u8 = x_dev.dtype == torch.uint8
        if not self._dp:
            # single GPU / fused data parallel: one call; the gradient-slab reduction rides in the optimizer launch
            fn = self._lib.ga3c_train_step_u8 if u8 else self._lib.ga3c_train_step
            _capi.check(fn(self._h, x_dev.data_ptr(), yr_dev.data_ptr(), a_dev.data_ptr(), b, float(self.learning_rate),
                           float(self.beta), loss_ptr, st.cuda_stream), "ga3c_train_step")
            return
        if b == 0:
            # lock-step tick of a rank with no experiences (threads.LockstepTrainer): zero contribution to the allreduce
            self._zero(self._grad_arena, st)
            if self._dual:
                self._zero(self._grad2_arena, st)
        elif self._dual:
            fb = self._lib.ga3c_dual_forward_backward_u8 if u8 else self._lib.ga3c_dual_forward_backward
            _capi.check(fb(self._h, x_dev.data_ptr(), yr_dev.data_ptr(), a_dev.data_ptr(), b, float(self.beta), loss_ptr,
                           st.cuda_stream), "ga3c_dual_forward_backward")
        if self._dual:
            for ar in (self._allreduce, self._allreduce2):
                ar.start_big(st)
                ar.finish(st)
            _capi.check(self._lib.ga3c_dual_apply(self._h, float(self.learning_rate), st.cuda_stream), "ga3c_dual_apply")
            return
        if b == 0:
            self._allreduce.start_big(st)
            self._allreduce.finish(st)
        else:
            # dense1/w (98.8 % of the arena) is final after the head: its allreduce overlaps the conv backward
            head = self._lib.ga3c_fb_head_u8 if u8 else self._lib.ga3c_fb_head
            tail = self._lib.ga3c_fb_tail_u8 if u8 else self._lib.ga3c_fb_tail
            _capi.check(head(self._h, x_dev.data_ptr(), yr_dev.data_ptr(), a_dev.data_ptr(), b,
                             float(self.beta), loss_ptr, st.cuda_stream), "ga3c_fb_head")
            self._allreduce.start_big(st)
            _capi.check(tail(self._h, x_dev.data_ptr(), b, st.cuda_stream), "ga3c_fb_tail")
            self._allreduce.finish(st)
        _capi.check(self._lib.ga3c_apply_rmsprop(self._h, float(self.learning_rate), st.cuda_stream), "ga3c_apply_rmsprop")

    @staticmethod
    def _zero(t: torch.Tensor, stream):
        with torch.cuda.stream(stream):
            t.zero_()

    def sync_replicas(self, src: int = 0):
        """Data parallel: make every rank's weights, RMSProp slots and step counter equal rank `src`'s (a collective: every
        rank calls it).  Run at construction, after load() and available after set_variables() / set_slots() with
        rank-dependent values."""
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1):
            return
        which = [0, 2, 3] + ([5, 6] if self._dual else [])
        for w in which:
            t = torch.from_numpy(self._download(w)).to(self._tdev)
            dist.broadcast(t, src=src)
            self._upload(w, t.cpu().numpy())
        step = torch.tensor([self.get_global_step()], dtype=torch.int64, device=self._tdev)
        dist.broadcast(step, src=src)
        self._lib.ga3c_set_global_step(self._h, int(step.item()))

    # ------------------------------------------------------------------ reference API (host numpy)
    def predict_p_and_v(self, x):
        """NetworkVP.py:248-252.  x: float32 [B, state_dim] (a view of the predictor's reused buffer,
        ThreadPredictor.py:57 -- consumed before returning).  Returns [p [B,A] f32, v [B] f32]."""
        x = np.asarray(x)
        if x.ndim != 2 or x.shape[1] != self.state_dim:
            raise ValueError(f"x must be [B, {self.state_dim}], got {x.shape}")
        x = self._frames(x, self.state_dim)
        b = x.shape[0]
        if b == 0:
            return [np.zeros((0, self.num_actions), np.float32), np.zeros((0,), np.float32)]
        with self._lock:
            self._ensure(b)
            hx, dx = self._io_u8() if x.dtype == np.uint8 else (self._hx, self._dx)
            with torch.cuda.stream(self._stream):
                self._h2d(x, hx, dx, b)
                self.predict_device(dx[:b], self._dp_out[:b], self._dv_out[:b], stream=self._stream)
                self._hp[:b].copy_(self._dp_out[:b], non_blocking=True)
                self._hv[:b].copy_(self._dv_out[:b], non_blocking=True)
            self._stream.synchronize()
            return [self._hp[:b].numpy().copy(), self._hv[:b].numpy().copy()]

    def train(self, x, y_r, a, x2=None, done=None, trainer_id=0, *, fetch_losses=False):
        """NetworkVP.py:254-257.  x2, done, trainer_id are accepted and ignored exactly as the A3C
        networks of the reference ignore them; y_r may arrive as float64 (ProcessAgent.py:99)."""
        x = np.asarray(x)
        b = x.shape[0]
        if b == 0:
            if self.dp_mode is None:
                return None
            # data parallel: every rank enters every step; an empty batch contributes a zero gradient (ga3c_train_step with
            # batch = 0) and this rank applies the same update as the others
            with self._lock:
                with torch.cuda.stream(self._stream):
                    self.train_device(self._dx[:0], self._dyr[:0], self._da[:0],
                                      loss_out=self._loss_dev if fetch_losses else None, stream=self._stream)
                self._stream.synchronize()
            self.dp_check()
            return dict(cost_p_1=0.0, cost_p_2=0.0, cost_p=0.0, cost_v=0.0, cost_all=0.0) if fetch_losses else None
        x = self._frames(x, self.state_dim)
        y_r = np.asarray(y_r, dtype=np.float32).reshape(b)
        a = np.asarray(a, dtype=np.float32).reshape(b, self.num_actions)
        slot = self._train_slots[int(trainer_id) % len(self._train_slots) if isinstance(trainer_id, (int, np.integer)) else 0]
        with slot.lock:
            # this call's inputs travel on the slot's stream, outside the handle lock: under the kernels of the other trainer's call
            hx, dx = slot.buffers(b, self.num_actions, x.dtype == np.uint8)
            with torch.cuda.stream(slot.stream):
                self._h2d(y_r, slot.hyr, slot.dyr, b)
                self._h2d(a, slot.ha, slot.da, b)
                self._h2d(x, hx, dx, b)
                slot.ready.record(slot.stream)
            with self._lock:
                self._ensure(b)
                self._stream.wait_event(slot.ready)
                with torch.cuda.stream(self._stream):
                    self.train_device(dx[:b], slot.dyr[:b], slot.da[:b],
                                      loss_out=self._loss_dev if fetch_losses else None, stream=self._stream)
                    losses = self._loss_dev.cpu() if fetch_losses else None
                self._stream.synchronize()
        if self.dp_mode == "fused":
            self._dp_steps = getattr(self, "_dp_steps", 0) + 1
            if self._dp_steps % 64 == 1:      # a timed-out cross-rank wait leaves garbage weights: fail, do not train on
                self.dp_check()
        if fetch_losses:
            self.last_losses = self._loss_dict(losses)
            return self.last_losses
        return None

    def losses(self, x, y_r, a):
        """Forward + loss only (what `log` evaluates, NetworkVP.py:259-265), without touching the weights:
        runs forward_backward and discards the gradients."""
        x = self._frames(x, self.state_dim)
        b = x.shape[0]
        with self._lock:
            self._ensure(b)
            st = self._stream
            with torch.cuda.stream(st):
                dx = torch.as_tensor(x, device=self._tdev)
                dyr = torch.as_tensor(np.asarray(y_r, dtype=np.float32).reshape(b), device=self._tdev)
                da = torch.as_tensor(np.asarray(a, dtype=np.float32).reshape(b, self.num_actions), device=self._tdev)
                fn = self._lib.ga3c_forward_backward_u8 if x.dtype == np.uint8 else self._lib.ga3c_forward_backward
                _capi.check(fn(self._h, dx.data_ptr(), dyr.data_ptr(), da.data_ptr(), b, float(self.beta),
                               self._loss_dev.data_ptr(), st.cuda_stream), "ga3c_forward_backward")
                l = self._loss_dev.cpu()
            st.synchronize()
        return self._loss_dict(l)

    # ------------------------------------------------------------------ TensorBoard summaries (NetworkVP.py:152-173, :259-265)
    def _summary_pass(self, x, y_r, a, loss_ptr, st):
        """predict, then forward_backward with the loss sums to loss_ptr, on st, for frames x (float32 or uint8); returns the
        rows.  predict goes first: it rewrites n2 / d1 of the workspace, which forward_backward then leaves as the training
        forward computes them.  Histogram tags: the 10 variables, then activation_n1, activation_n2, activation_d2 (dense1),
        activation_v and activation_p; n1 and n2 are histogrammed as the network stores them (bf16)."""
        x = self._frames(x, self.state_dim)
        b = x.shape[0]
        y_r = np.asarray(y_r, dtype=np.float32).reshape(b)
        a = np.asarray(a, dtype=np.float32).reshape(b, self.num_actions)
        u8 = x.dtype == np.uint8
        self._ensure(b)
        hx, dx = self._io_u8() if u8 else (self._hx, self._dx)
        self._h2d(x, hx, dx, b)
        self._h2d(y_r, self._hyr, self._dyr, b)
        self._h2d(a, self._ha, self._da, b)
        pred = self._lib.ga3c_predict_u8 if u8 else self._lib.ga3c_predict
        _capi.check(pred(self._h, dx.data_ptr(), b, self._dp_out.data_ptr(), self._dv_out.data_ptr(), st.cuda_stream),
                    "ga3c_predict")
        fb = self._lib.ga3c_forward_backward_u8 if u8 else self._lib.ga3c_forward_backward
        _capi.check(fb(self._h, dx.data_ptr(), self._dyr.data_ptr(), self._da.data_ptr(), b, float(self.beta), loss_ptr,
                       st.cuda_stream), "ga3c_forward_backward")
        return b

    def log(self, x, y_r, a, training_step, feed_dict=None):
        """NetworkVP.py:259-265: appends the six scalars to logs/<model_name>/scalars.csv (as the MLP networks do) and writes
        them with the 15 histograms of `histograms` at step `training_step` to a TensorBoard event file in logs/<model_name>
        (needs the optional tensorboard package; without it: the CSV line and one warning).  A NaN / Inf in a histogram raises
        ValueError naming its tag after the CSV line is written; no event is written for that call.  With the peer-memory
        data-parallel exchange (dp_mode 'fused') the dense1/w slices live on their owners: CSV only, one warning."""
        if self.dp_mode == "fused":
            if not getattr(self, "_warned_fused_log", False):
                self._warned_fused_log = True
                warnings.warn("Network.log: no TensorBoard histograms with dp_mode 'fused'; writing scalars.csv only",
                              RuntimeWarning, stacklevel=2)
            return super().log(x, y_r, a, training_step, feed_dict)
        self._log_summaries(*self._summaries(x, y_r, a), training_step)

    # ------------------------------------------------------------------ variables / checkpoints
    def _download(self, which: int) -> np.ndarray:
        self.dp_check()
        return super()._download(which)

    def get_gradients(self):
        """Gradients left by the last forward_backward.  Data parallel: dp_mode 'nccl' leaves the allreduced gradient on every
        rank; dp_mode 'fused' leaves this rank's OWN contribution, except for the slice of dense1/w this rank owns, which
        holds the sum over ranks (the reduction happens on the owner; only the bf16 shadow of the new weights travels)."""
        return self._split(self._download(1))

    def _after_load(self):
        if self.dp_mode is not None:
            self.sync_replicas()          # every rank read the same file; make sure of it

    def dp_check(self):
        """Raises if a cross-rank wait of the data-parallel exchange gave up (a rank died or the ranks' train() calls fell
        out of step): every such wait is bounded so that nothing hangs, but the replicas are no longer in sync."""
        err = C.c_int32(0)
        _capi.check(self._lib.ga3c_dp_error(self._h, C.byref(err)), "ga3c_dp_error")
        if err.value:
            raise _capi.Ga3cError(f"data-parallel exchange timed out waiting for a peer rank (wait bits {err.value:#x}, "
                                  "dp_exchange.cuh): replicas are out of sync")

    # ------------------------------------------------------------------ introspection (tests / profiling)
    def trace_begin(self, stream=None):
        """Start a step timeline trace (ga3c_trace_begin): kernels stamp %globaltimer at launch / start / end."""
        st = stream if stream is not None else torch.cuda.current_stream(self._tdev)
        _capi.check(self._lib.ga3c_trace_begin(self._h, st.cuda_stream), "ga3c_trace_begin")

    def trace_end(self) -> dict:
        """{kernel name: (first launched, last launched, first started, last started, first ended, last ended)} in
        microseconds relative to the earliest stamp; kernels that did not run are omitted.  Synchronises."""
        n = self._lib.ga3c_kernel_count()
        buf = (C.c_uint64 * (6 * n))()
        _capi.check(self._lib.ga3c_trace_end(self._h, buf, n), "ga3c_trace_end")
        rows = {self._lib.ga3c_kernel_name(k).decode(): [buf[6 * k + i] for i in range(6)] for k in range(n)}
        rows = {k: v for k, v in rows.items() if v[1] != 0}
        t0 = min(v[0] for v in rows.values()) if rows else 0
        return {k: tuple((t - t0) / 1e3 for t in v) for k, v in rows.items()}

    def keep_dn1(self, on: bool):
        """Tests: make the fused conv backward also store dn1 (normally shared-memory only) to the workspace."""
        _capi.check(self._lib.ga3c_keep_dn1(self._h, int(bool(on))), "ga3c_keep_dn1")

    def workspace(self, which: int) -> np.ndarray:
        """Activation workspace of the last call as float32 numpy (bf16 buffers are widened), flat in the LOGICAL order of the
        reference tensors: n1 (0) and dn2 (4) live in HBM in the tcgen05 operand layouts the conv backward consumes
        (include/ga3c_b200.h, ga3c_workspace_ptr) and are unscrambled here to [B, 21*21*16] / [B, 11*11*32]; 7 = the bf16 copy of
        the frames, unscrambled to the padded image [B, 88, 88, 4].  Any other geometry than 84x84x4 keeps them row-major: n1 and
        dn1 [B, H1*W1*16], n2 and dn2 [B, H2*W2*32], 7 the im2col matrix of the frames [B*H1*W1, 64C + 8]."""
        ptr, nbytes = C.c_void_p(), C.c_int64()
        _capi.check(self._lib.ga3c_workspace_ptr(self._h, which, C.byref(ptr), C.byref(nbytes)), "ga3c_workspace_ptr")
        torch.cuda.synchronize(self._tdev)
        if which == 2:
            t = torch.as_tensor(_DevArray(ptr.value, nbytes.value // 4, self), device=self._tdev)
            return t.cpu().numpy().copy()
        iface = {"shape": (nbytes.value // 2,), "typestr": "<i2", "data": (ptr.value, False), "version": 2}
        holder = type("H", (), {"__cuda_array_interface__": iface})()
        t = torch.as_tensor(holder, device=self._tdev).view(torch.bfloat16)
        flat = t.float().cpu().numpy().copy()
        if self.geometry != (84, 84, 4):
            return flat
        if which == 0:            # Blk2: [B][plane = ((Y&1)*2 + (X&1))*2 + h][row = (Y>>1)*13 + (X>>1)][8], Y = y + 1, X = x + 1
            raw = flat.reshape(-1, 8, 160, 8)
            y, x, h = np.meshgrid(np.arange(21), np.arange(21), np.arange(2), indexing="ij")
            plane = (((y + 1) & 1) * 2 + ((x + 1) & 1)) * 2 + h
            row = ((y + 1) >> 1) * 13 + ((x + 1) >> 1)
            return raw[:, plane, row, :].reshape(raw.shape[0], -1).ravel()         # [B, y, x, h, 8] = [B, 441 * 16]
        if which == 4:            # G: [B][plane j][row = (oy+1)*13 + ox+1][8]
            raw = flat.reshape(-1, 4, 172, 8)
            oy, ox, j = np.meshgrid(np.arange(11), np.arange(11), np.arange(4), indexing="ij")
            return raw[:, j, (oy + 1) * 13 + ox + 1, :].reshape(raw.shape[0], -1).ravel()   # [B, oy, ox, j, 8] = [B, 3872]
        if which == 7:            # xblk: [B][quarter][plane = dy*2 + (dx>>1)][128 rows][(dx&1, c)], block row = Y*22 + X
            raw = flat.reshape(-1, 4, 8, 128, 8)
            py, px, c = np.meshgrid(np.arange(88), np.arange(88), np.arange(4), indexing="ij")
            r = (py >> 2) * 22 + (px >> 2)
            plane = (py & 3) * 2 + ((px & 3) >> 1)
            return raw[:, r >> 7, plane, r & 127, (px & 1) * 4 + c].reshape(raw.shape[0], -1).ravel()
        return flat
