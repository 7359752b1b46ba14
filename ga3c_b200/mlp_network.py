"""Drop-ins for the fork's two low-dimensional `Network` plugins (BASELINE config 4; SURVEY 8a rows A6 / A7):

    NetworkVP            fork NetworkVP.py:36-288      x[S] -> 4 -> 256 -> 256 (linear) -> 100 -> 64 (sigmoid); value head +
                                                       atan2 angle head; softmax_p = log_softmax_p = logits_p (:95-96)
    NetworkVP_discrate   NetworkVP_discrate.py:36-130  Config.DENSE_LAYERS all built from x (:55, as written: only the last one
                                                       is live); softmax / A3C loss heads (:60-85)

Same constructor, attributes and methods as the reference classes (see ga3c_b200.network.Network for the conv net).  Every
kernel is launched by the C-ABI library (ga3c_mlp_*, include/ga3c_b200.h); PyTorch holds buffers and the stream only.  No
CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os
import re
import threading

import numpy as np
import torch

from . import _capi, summaries
from ._arena import ArenaNetworkMixin
from .config import Config as _DefaultConfig
from .network import _parse_device


class _MlpNetwork(ArenaNetworkMixin):
    KIND = None

    def __init__(self, device, model_name, num_actions, state_dim, *, config=None, max_batch=None, seed=None):
        cfg = config or _DefaultConfig
        self.config = cfg
        self.device = device
        self.model_name = model_name
        self.num_actions = int(num_actions)
        self.state_dim = int(np.prod(state_dim)) if not isinstance(state_dim, int) else state_dim
        self._dual = bool(getattr(cfg, "DUAL_RMSPROP", False))
        self.learning_rate = cfg.LEARNING_RATE_START
        self.beta = cfg.BETA_START
        self.log_epsilon = cfg.LOG_EPSILON

        self._lib = _capi.load()
        if not torch.cuda.is_available():
            raise _capi.Ga3cError("no CUDA device visible: ga3c_b200 has no CPU fallback")
        self._ordinal = _parse_device(device)
        self._tdev = torch.device("cuda", self._ordinal)
        self._lock = threading.Lock()
        self._max_batch = int(max_batch or max(getattr(cfg, "PREDICTION_BATCH_SIZE", 128), 128))
        dense = tuple(getattr(cfg, "DENSE_LAYERS", (10, 10, 10, 10)))          # Config.py:107
        c = _capi.ga3c_mlp_config(device=self._ordinal, kind=self.KIND, state_dim=self.state_dim,
                                  num_actions=self.num_actions, max_batch=self._max_batch, n_dense=len(dense),
                                  dense_width=(C.c_int32 * 8)(*dense[:8]),
                                  rmsprop_decay=cfg.RMSPROP_DECAY, rmsprop_momentum=cfg.RMSPROP_MOMENTUM,
                                  rmsprop_epsilon=cfg.RMSPROP_EPSILON, log_epsilon=cfg.LOG_EPSILON,
                                  min_policy=cfg.MIN_POLICY,
                                  use_log_softmax=int(bool(getattr(cfg, 'USE_LOG_SOFTMAX', False))),
                              use_grad_clip=int(bool(getattr(cfg, 'USE_GRAD_CLIP', False))),
                              grad_clip_norm=float(getattr(cfg, 'GRAD_CLIP_NORM', 40.0)), dual_rmsprop=int(self._dual))
        if self.KIND == _capi.MLP_DISCRATE and len(dense) > 8:
            raise ValueError("Config.DENSE_LAYERS: at most 8 entries")
        h = C.c_void_p()
        _capi.check(self._lib.ga3c_mlp_create(C.byref(c), C.byref(h)), "ga3c_mlp_create")
        self._h = h

        self._table, self._live = {}, {}
        for i in range(self._lib.ga3c_mlp_param_count(self._h)):
            name, off, nd, live = C.c_char_p(), C.c_int64(), C.c_int32(), C.c_int32()
            shape = (C.c_int64 * 4)()
            _capi.check(self._lib.ga3c_mlp_param_info(self._h, i, C.byref(name), C.byref(off), C.byref(nd), shape,
                                                      C.byref(live)), "ga3c_mlp_param_info")
            self._table[name.value.decode()] = (off.value, tuple(shape[k] for k in range(nd.value)))
            self._live[name.value.decode()] = bool(live.value)
        self._arena_floats = self._lib.ga3c_mlp_arena_floats(self._h)
        with torch.cuda.device(self._tdev):
            self._stream = torch.cuda.Stream(device=self._tdev)
            self._loss_dev = torch.zeros(4, dtype=torch.float32, device=self._tdev)
        self._alloc_io(self._max_batch)

        # every variable: U(-0.3, 0.3)  (dense_layer, NetworkVP.py:199-202)
        rng = np.random.default_rng(seed)
        self.set_variables({k: rng.uniform(-0.3, 0.3, size=s).astype(np.float32) for k, (_, s) in self._table.items()})
        self.last_losses = None
        self._hist_tags = summaries.mlp_histogram_tags([(k, self._live[k]) for k in self._table])
        if len(self._hist_tags) != self._lib.ga3c_mlp_histogram_count(self._h):
            raise _capi.Ga3cError("ga3c_mlp_histogram_count disagrees with the variable table")
        self._summ_dev = self._summ_host = None     # log / histograms: device results and their pinned copy
        self._events = None                         # the TensorBoard event file, opened by the first log()

    # ------------------------------------------------------------------ buffers
    def _alloc_io(self, rows: int):
        a, s = self.num_actions, self.state_dim
        with torch.cuda.device(self._tdev):
            self._hx = torch.empty((rows, s), dtype=torch.float32, pin_memory=True)
            self._hyr = torch.empty((rows,), dtype=torch.float32, pin_memory=True)
            self._ha = torch.empty((rows, a), dtype=torch.float32, pin_memory=True)
            self._hp = torch.empty((rows, a), dtype=torch.float32, pin_memory=True)
            self._hv = torch.empty((rows,), dtype=torch.float32, pin_memory=True)
            self._dx = torch.empty((rows, s), dtype=torch.float32, device=self._tdev)
            self._dyr = torch.empty((rows,), dtype=torch.float32, device=self._tdev)
            self._da = torch.empty((rows, a), dtype=torch.float32, device=self._tdev)
            self._dp_out = torch.empty((rows, a), dtype=torch.float32, device=self._tdev)
            self._dv_out = torch.empty((rows,), dtype=torch.float32, device=self._tdev)
        self._io_rows = rows

    def _ensure(self, rows: int):
        if rows > self._max_batch:
            _capi.check(self._lib.ga3c_mlp_reserve(self._h, rows), "ga3c_mlp_reserve")
            self._max_batch = rows
        if rows > self._io_rows:
            self._alloc_io(rows)

    def __del__(self):
        try:
            if getattr(self, "_events", None) is not None:
                self._events.close()
            if getattr(self, "_h", None):
                self._lib.ga3c_mlp_destroy(self._h)
                self._h = None
        except Exception:
            pass

    # ------------------------------------------------------------------ device-resident API
    def predict_device(self, x_dev, p_out=None, v_out=None, stream=None):
        b = x_dev.shape[0]
        self._ensure(b)
        if p_out is None:
            p_out = torch.empty((b, self.num_actions), dtype=torch.float32, device=self._tdev)
        if v_out is None:
            v_out = torch.empty((b,), dtype=torch.float32, device=self._tdev)
        st = stream or torch.cuda.current_stream(self._tdev)
        _capi.check(self._lib.ga3c_mlp_predict(self._h, x_dev.data_ptr(), b, p_out.data_ptr(), v_out.data_ptr(),
                                               st.cuda_stream), "ga3c_mlp_predict")
        return p_out, v_out

    def train_device(self, x_dev, yr_dev, a_dev, *, loss_out=None, stream=None):
        b = x_dev.shape[0]
        self._ensure(b)
        st = stream or torch.cuda.current_stream(self._tdev)
        _capi.check(self._lib.ga3c_mlp_train_step(self._h, x_dev.data_ptr(), yr_dev.data_ptr(), a_dev.data_ptr(), b,
                                                  float(self.learning_rate), float(self.beta),
                                                  loss_out.data_ptr() if loss_out is not None else None, st.cuda_stream),
                    "ga3c_mlp_train_step")

    def forward_backward_device(self, x_dev, yr_dev, a_dev, *, loss_out=None, stream=None):
        b = x_dev.shape[0]
        self._ensure(b)
        st = stream or torch.cuda.current_stream(self._tdev)
        _capi.check(self._lib.ga3c_mlp_forward_backward(self._h, x_dev.data_ptr(), yr_dev.data_ptr(), a_dev.data_ptr(), b,
                                                        float(self.beta),
                                                        loss_out.data_ptr() if loss_out is not None else None,
                                                        st.cuda_stream), "ga3c_mlp_forward_backward")

    # ------------------------------------------------------------------ reference API (host numpy)
    def _rows(self, x):
        x = np.asarray(x, dtype=np.float32)
        if x.ndim != 2 or x.shape[1] != self.state_dim:
            raise ValueError(f"x must be [B, {self.state_dim}], got {x.shape}")
        return x

    def predict_p_and_v(self, x):
        """NetworkVP.py:248-252 -> [softmax_p [B,A] f32, logits_v [B] f32]."""
        x = self._rows(x)
        b = x.shape[0]
        if b == 0:
            return [np.zeros((0, self.num_actions), np.float32), np.zeros((0,), np.float32)]
        with self._lock:
            self._ensure(b)
            self._hx[:b].numpy()[...] = x
            with torch.cuda.stream(self._stream):
                self._dx[:b].copy_(self._hx[:b], non_blocking=True)
                self.predict_device(self._dx[:b], self._dp_out[:b], self._dv_out[:b], stream=self._stream)
                self._hp[:b].copy_(self._dp_out[:b], non_blocking=True)
                self._hv[:b].copy_(self._dv_out[:b], non_blocking=True)
            self._stream.synchronize()
            return [self._hp[:b].numpy().copy(), self._hv[:b].numpy().copy()]

    def _stage_train(self, x, y_r, a):
        x = self._rows(x)
        b = x.shape[0]
        self._ensure(b)
        self._hx[:b].numpy()[...] = x
        self._hyr[:b].numpy()[...] = np.asarray(y_r, dtype=np.float32).reshape(b)
        self._ha[:b].numpy()[...] = np.asarray(a, dtype=np.float32).reshape(b, self.num_actions)
        self._dx[:b].copy_(self._hx[:b], non_blocking=True)
        self._dyr[:b].copy_(self._hyr[:b], non_blocking=True)
        self._da[:b].copy_(self._ha[:b], non_blocking=True)
        return b

    @staticmethod
    def _loss_dict(l):
        c1, c2, cv = (float(v) for v in l[:3])
        return dict(cost_p_1=c1, cost_p_2=c2, cost_p=-(c1 + c2), cost_v=cv, cost_all=-(c1 + c2) + cv)

    def train(self, x, y_r, a, x2=None, done=None, trainer_id=0, *, fetch_losses=False):
        """NetworkVP.py:254-257; x2, done, trainer_id are ignored as in the reference."""
        if np.asarray(x).shape[0] == 0:
            return None
        with self._lock:
            with torch.cuda.stream(self._stream):
                b = self._stage_train(x, y_r, a)
                self.train_device(self._dx[:b], self._dyr[:b], self._da[:b],
                                  loss_out=self._loss_dev if fetch_losses else None, stream=self._stream)
                losses = self._loss_dev.cpu() if fetch_losses else None
            self._stream.synchronize()
        if fetch_losses:
            self.last_losses = self._loss_dict(losses)
            return self.last_losses
        return None

    def losses(self, x, y_r, a):
        """Forward + loss (what `log` evaluates) without touching the weights; leaves the gradients in the gradient arena."""
        with self._lock:
            with torch.cuda.stream(self._stream):
                b = self._stage_train(x, y_r, a)
                self.forward_backward_device(self._dx[:b], self._dyr[:b], self._da[:b], loss_out=self._loss_dev,
                                             stream=self._stream)
                l = self._loss_dev.cpu()
            self._stream.synchronize()
        return self._loss_dict(l)

    # ------------------------------------------------------------------ TensorBoard summaries (NetworkVP.py:152-173, :259-265)
    _HROW = 5 + summaries.BUCKETS

    def _summaries(self, x, y_r, a):
        """predict, forward_backward and ga3c_mlp_histograms on the same rows as ONE critical section of the handle (no trainer
        thread can overwrite the layer outputs in between), then one device -> host copy.  predict goes first: for a
        tensor-core batch it writes its layer outputs through the training workspace, which forward_backward then rewrites.
        Weights, slots and the step counter are not touched.  Returns (losses, {tag: (min, max, num, sum, sum_squares,
        counts)}, [tags of the histograms holding a NaN / Inf])."""
        x = self._rows(x)
        if x.shape[0] == 0:
            raise ValueError("the summaries need at least one row")
        tags = self._hist_tags
        n_hist = len(tags) * self._HROW
        n_bad = (len(tags) + 1) // 2
        if self._summ_dev is None:
            # [histogram rows | int32 non-finite flags | 4 fp32 loss sums] as doubles, so that one copy brings it all back
            with torch.cuda.device(self._tdev):
                self._summ_dev = torch.empty(n_hist + n_bad + 2, dtype=torch.float64, device=self._tdev)
                self._summ_host = torch.empty(n_hist + n_bad + 2, dtype=torch.float64, pin_memory=True)
        base = self._summ_dev.data_ptr()
        bad_ptr, loss_ptr = base + 8 * n_hist, base + 8 * (n_hist + n_bad)
        with self._lock:
            st = self._stream
            with torch.cuda.stream(st):
                b = self._stage_train(x, y_r, a)
                dx, dp, dv = self._dx[:b], self._dp_out[:b], self._dv_out[:b]
                self.predict_device(dx, dp, dv, stream=st)
                _capi.check(self._lib.ga3c_mlp_forward_backward(self._h, dx.data_ptr(), self._dyr.data_ptr(), self._da.data_ptr(),
                                                                b, float(self.beta), loss_ptr, st.cuda_stream),
                            "ga3c_mlp_forward_backward")
                _capi.check(self._lib.ga3c_mlp_histograms(self._h, b, dp.data_ptr(), dv.data_ptr(), base, bad_ptr,
                                                          st.cuda_stream), "ga3c_mlp_histograms")
                self._summ_host.copy_(self._summ_dev, non_blocking=True)
            st.synchronize()
            host = self._summ_host.numpy().copy()
        rows = host[:n_hist].reshape(len(tags), self._HROW)
        stats = {t: (r[0], r[1], r[2], r[3], r[4], r[5:]) for t, r in zip(tags, rows)}
        bad = host[n_hist:n_hist + n_bad].view(np.int32)[:len(tags)]
        l = self._loss_dict(host[n_hist + n_bad:].view(np.float32))
        return l, stats, [t for t, f in zip(tags, bad) if f]

    def histograms(self, x, y_r, a) -> dict:
        """The histograms `log` writes, for rows x [B, S] and targets y_r, a: {tag: (min, max, num, sum, sum_squares, counts)},
        TF's histogram::Histogram with its 1551 default buckets (ga3c_b200.summaries.LIMITS), computed on the GPU.  Tags
        (summaries.mlp_histogram_tags): weights_<variable name> (tf.summary's tag cleaning, e.g. weights_dense1/w_0) for every
        variable in TF creation order, gradient-less ones included; activation_<layer scope> for every live hidden layer in
        forward order (fork NetworkVP: activation_dense11_p ... activation_dense14_p, activation_dense1; NetworkVP_discrate:
        activation_dense1_<n>_p); then activation_v (logits_v) and activation_p (softmax_p: for the fork NetworkVP the atan2
        output).  Raises ValueError on a NaN / Inf."""
        _, stats, bad = self._summaries(x, y_r, a)
        if bad:
            raise self._nonfinite(bad)
        return stats

    def log(self, x, y_r, a, training_step, feed_dict=None):
        """NetworkVP.py:259-265: appends the six scalars to logs/<model_name>/scalars.csv and writes them with the histograms
        of `histograms` at step `training_step` to a TensorBoard event file in logs/<model_name> (needs the optional
        tensorboard package; without it: the CSV line and one warning).  A NaN / Inf in a histogram raises ValueError naming
        its tag after the CSV line is written; no event is written for that call."""
        self._log_summaries(*self._summaries(x, y_r, a), training_step)

    # ------------------------------------------------------------------ variables / checkpoints
    def get_global_step(self):
        return int(self._lib.ga3c_mlp_global_step(self._h))

    def live_variables(self):
        return [k for k in self._table if self._live[k]]

    def _download(self, which: int) -> np.ndarray:
        out = np.empty(self._arena_floats, dtype=np.float32)
        with self._lock:
            _capi.check(self._lib.ga3c_mlp_arena_download(self._h, which, out.ctypes.data, out.size), "ga3c_mlp_arena_download")
        return out

    def _upload(self, which: int, arena: np.ndarray):
        arena = np.ascontiguousarray(arena, dtype=np.float32)
        with self._lock:
            _capi.check(self._lib.ga3c_mlp_arena_upload(self._h, which, arena.ctypes.data, arena.size), "ga3c_mlp_arena_upload")

    def get_gradients(self):
        """Gradients of the last forward_backward; live variables only (the others have none)."""
        g = self._split(self._download(1))
        return {k: v for k, v in g.items() if self._live[k]}

    def _set_global_step(self, step: int):
        self._lib.ga3c_mlp_set_global_step(self._h, int(step))

    # ------------------------------------------------------------------ introspection
    def workspace(self, which: int, layer: int, batch: int) -> np.ndarray:
        """Parity tests: output (which = 0) or pre-activation gradient (1) of live hidden layer `layer` for the first `batch`
        rows of the last forward/backward, as a host array."""
        ptr, width = C.c_void_p(), C.c_int32()
        _capi.check(self._lib.ga3c_mlp_workspace_ptr(self._h, int(which), int(layer), C.byref(ptr), C.byref(width)),
                    "ga3c_mlp_workspace_ptr")
        torch.cuda.synchronize(self._tdev)
        iface = {"shape": (int(batch) * width.value,), "typestr": "<f4", "data": (ptr.value, False), "version": 2}
        holder = type("H", (), {"__cuda_array_interface__": iface})()
        return torch.as_tensor(holder, device=self._tdev).cpu().numpy().reshape(int(batch), width.value).copy()

    def launch_count(self) -> int:
        return int(self._lib.ga3c_mlp_launch_count(self._h))

    def kernel_timing(self, max_records: int):
        _capi.check(self._lib.ga3c_mlp_timing_enable(self._h, int(max_records)), "ga3c_mlp_timing_enable")

    def kernel_times(self) -> dict:
        n = self._lib.ga3c_kernel_count()
        tot, cnt = (C.c_double * n)(), (C.c_int64 * n)()
        _capi.check(self._lib.ga3c_mlp_timing_collect(self._h, tot, cnt, n), "ga3c_mlp_timing_collect")
        return {self._lib.ga3c_kernel_name(k).decode(): (tot[k], cnt[k]) for k in range(n) if cnt[k]}


class NetworkVP(_MlpNetwork):
    """The fork's NetworkVP.py `Network` (Pendulum / pyperrace: S = 3 or 4, A = 1 or 2)."""
    KIND = _capi.MLP_FORK_VP


class NetworkVP_discrate(_MlpNetwork):
    """NetworkVP_discrate.py `Network` (CartPole: S = 4, A = 2, Config.DENSE_LAYERS = (10, 10, 10, 10))."""
    KIND = _capi.MLP_DISCRATE
