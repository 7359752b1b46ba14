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
import threading

import numpy as np
import torch

from . import _capi, summaries
from ._arena import ArenaNetworkMixin
from .config import Config as _DefaultConfig


class _MlpNetwork(ArenaNetworkMixin):
    KIND = None
    _PREFIX = "ga3c_mlp_"

    def __init__(self, device, model_name, num_actions, state_dim, *, config=None, max_batch=None, seed=None):
        cfg = config or _DefaultConfig
        fields = self._setup(device, model_name, num_actions, state_dim, cfg, max_batch)
        self._lock = threading.Lock()
        dense = tuple(getattr(cfg, "DENSE_LAYERS", (10, 10, 10, 10)))          # Config.py:107
        c = _capi.ga3c_mlp_config(device=self._ordinal, kind=self.KIND, state_dim=self.state_dim,
                                  num_actions=self.num_actions, max_batch=self._max_batch, n_dense=len(dense),
                                  dense_width=(C.c_int32 * 8)(*dense[:8]), **fields)
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
        self._hist_tags = summaries.mlp_histogram_tags([(k, self._live[k]) for k in self._table])
        if len(self._hist_tags) != self._lib.ga3c_mlp_histogram_count(self._h):
            raise _capi.Ga3cError("ga3c_mlp_histogram_count disagrees with the variable table")

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
    def _summary_pass(self, x, y_r, a, loss_ptr, st):
        """predict, then forward_backward with the loss sums to loss_ptr, on st; returns the rows.  predict goes first: for a
        tensor-core batch it writes its layer outputs through the training workspace, which forward_backward then rewrites.
        Histogram tags (summaries.mlp_histogram_tags): every variable, gradient-less ones included; activation_<layer scope>
        for every live hidden layer in forward order (fork NetworkVP: activation_dense11_p ... activation_dense14_p,
        activation_dense1; NetworkVP_discrate: activation_dense1_<n>_p); activation_v (logits_v) and activation_p (softmax_p:
        for the fork NetworkVP the atan2 output)."""
        b = self._stage_train(x, y_r, a)
        dx = self._dx[:b]
        self.predict_device(dx, self._dp_out[:b], self._dv_out[:b], stream=st)
        self._call("forward_backward", dx.data_ptr(), self._dyr.data_ptr(), self._da.data_ptr(), b, float(self.beta),
                   loss_ptr, st.cuda_stream)
        return b

    def log(self, x, y_r, a, training_step, feed_dict=None):
        """NetworkVP.py:259-265: appends the six scalars to logs/<model_name>/scalars.csv and writes them with the histograms
        of `histograms` at step `training_step` to a TensorBoard event file in logs/<model_name> (needs the optional
        tensorboard package; without it: the CSV line and one warning).  A NaN / Inf in a histogram raises ValueError naming
        its tag after the CSV line is written; no event is written for that call."""
        self._log_summaries(*self._summaries(x, y_r, a), training_step)

    # ------------------------------------------------------------------ variables / checkpoints
    def live_variables(self):
        return [k for k in self._table if self._live[k]]

    def get_gradients(self):
        """Gradients of the last forward_backward; live variables only (the others have none)."""
        g = self._split(self._download(1))
        return {k: v for k, v in g.items() if self._live[k]}

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


class NetworkVP(_MlpNetwork):
    """The fork's NetworkVP.py `Network` (Pendulum / pyperrace: S = 3 or 4, A = 1 or 2)."""
    KIND = _capi.MLP_FORK_VP


class NetworkVP_discrate(_MlpNetwork):
    """NetworkVP_discrate.py `Network` (CartPole: S = 4, A = 2, Config.DENSE_LAYERS = (10, 10, 10, 10))."""
    KIND = _capi.MLP_DISCRATE
