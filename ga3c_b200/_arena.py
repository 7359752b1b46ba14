"""What the conv `Network` and the low-dimensional MLP networks share on the host side: the reference's small accessors, the
flat parameter arena seen as a dict of TF-named tensors, RMSProp slots, checkpoints, the scalar log and the writing of
`log`'s TensorBoard event file; and, over the C ABI, the constructor prologue, the host staging buffers, the arena copies,
the summaries pass and the step counter / launch count / kernel timing.

The accessors, checkpoints and the scalar log need only `_table` ({TF variable name: (offset, shape)} into the fp32 arena, in
TF creation order), `_download(which)` / `_upload(which, arena)` (arena ids: 0 weights, 1 gradients, 2 / 3 ms / mom of the
first optimizer, 5 / 6 of the second), `get_global_step()`, `_set_global_step(step)`, `losses(x, y_r, a)`, and the
attributes `model_name`, `config`, `_dual`, `learning_rate`, `beta`.  The C-ABI methods call the library's functions named
`_PREFIX` + what they do (ga3c_arena_download / ga3c_mlp_arena_download, ...) on the handle `_h`.
"""
from __future__ import annotations

import ctypes as C
import os
import re

import numpy as np
import torch

from . import _capi, summaries


def _parse_device(device) -> int:
    """Config.DEVICE is a TF-style string 'gpu:0' (Config.py:62); 'cuda:0' and ints are accepted too."""
    if isinstance(device, int):
        return device
    m = re.fullmatch(r"/?(?:device:)?(gpu|cuda)(?::(\d+))?", str(device).strip().lower())
    if not m:
        raise ValueError(f"unsupported device {device!r}: this implementation is GPU-only ('gpu:N')")
    return int(m.group(2) or 0)


class ArenaNetworkMixin:
    _PREFIX = "ga3c_"
    _HROW = 5 + summaries.BUCKETS               # one histogram: min, max, num, sum, sum_squares, bucket counts

    # ------------------------------------------------------------------ the C ABI
    def _call(self, name: str, *args):
        fn = self._PREFIX + name
        _capi.check(getattr(self._lib, fn)(self._h, *args), fn)

    def _setup(self, device, model_name, num_actions, state_dim, cfg, max_batch) -> dict:
        """The constructor's first part: the reference's attributes, the library, the device and the workspace rows.  Returns
        the fields both config structs of the C ABI take from Config (optimizer, loss, gradient clipping)."""
        self.config = cfg
        self.device = device
        self.model_name = model_name
        self.num_actions = int(num_actions)
        self.state_dim = int(np.prod(state_dim)) if not isinstance(state_dim, int) else state_dim
        self._dual = bool(getattr(cfg, "DUAL_RMSPROP", False))
        self.learning_rate = cfg.LEARNING_RATE_START      # NetworkVP.py:44
        self.beta = cfg.BETA_START                        # NetworkVP.py:45
        self.log_epsilon = cfg.LOG_EPSILON                # NetworkVP.py:46
        self.last_losses = None
        self._summ_dev = self._summ_host = None           # log / histograms: device results and their pinned copy
        self._events = None                               # the TensorBoard event file, opened by the first log()

        self._lib = _capi.load()
        if not torch.cuda.is_available():
            raise _capi.Ga3cError("no CUDA device visible: ga3c_b200 has no CPU fallback")
        self._ordinal = _parse_device(device)
        self._tdev = torch.device("cuda", self._ordinal)
        self._max_batch = int(max_batch or max(getattr(cfg, "PREDICTION_BATCH_SIZE", 128), 128))
        return dict(rmsprop_decay=cfg.RMSPROP_DECAY, rmsprop_momentum=cfg.RMSPROP_MOMENTUM,
                    rmsprop_epsilon=cfg.RMSPROP_EPSILON, log_epsilon=cfg.LOG_EPSILON, min_policy=cfg.MIN_POLICY,
                    use_log_softmax=int(bool(getattr(cfg, 'USE_LOG_SOFTMAX', False))),
                    use_grad_clip=int(bool(getattr(cfg, 'USE_GRAD_CLIP', False))),
                    grad_clip_norm=float(getattr(cfg, 'GRAD_CLIP_NORM', 40.0)), dual_rmsprop=int(self._dual))

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
            self._call("reserve", rows)
            self._max_batch = rows
        if rows > self._io_rows:
            self._alloc_io(rows)

    def __del__(self):
        try:
            if getattr(self, "_events", None) is not None:
                self._events.close()
            if getattr(self, "_h", None):
                getattr(self._lib, self._PREFIX + "destroy")(self._h)
                self._h = None
        except Exception:
            pass

    def _download(self, which: int) -> np.ndarray:
        out = np.empty(self._arena_floats, dtype=np.float32)
        with self._lock:
            self._call("arena_download", which, out.ctypes.data, out.size)
        return out

    def _upload(self, which: int, arena: np.ndarray):
        arena = np.ascontiguousarray(arena, dtype=np.float32)
        with self._lock:
            self._call("arena_upload", which, arena.ctypes.data, arena.size)

    def get_global_step(self):              # NetworkVP.py:233-235
        return int(getattr(self._lib, self._PREFIX + "global_step")(self._h))

    def _set_global_step(self, step: int):
        getattr(self._lib, self._PREFIX + "set_global_step")(self._h, int(step))

    @staticmethod
    def _loss_dict(l):
        """The device's loss sums {cost_p_1, cost_p_2, cost_v, 0} as the reference's five costs."""
        c1, c2, cv = (float(v) for v in l[:3])
        return dict(cost_p_1=c1, cost_p_2=c2, cost_p=-(c1 + c2), cost_v=cv, cost_all=-(c1 + c2) + cv)

    # ------------------------------------------------------------------ TensorBoard summaries (NetworkVP.py:152-173, :259-265)
    def _summaries(self, x, y_r, a):
        """predict, forward_backward (`_summary_pass`) and the histograms on the same rows as ONE critical section of the
        handle (no trainer thread can overwrite the layer outputs in between), then one device -> host copy.  Weights, slots
        and the step counter are not touched.  Returns (losses, {tag: (min, max, num, sum, sum_squares, counts)}, [tags of
        the histograms holding a NaN / Inf])."""
        if len(x) == 0:
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
                b = self._summary_pass(x, y_r, a, loss_ptr, st)
                self._call("histograms", b, self._dp_out.data_ptr(), self._dv_out.data_ptr(), base, bad_ptr, st.cuda_stream)
                self._summ_host.copy_(self._summ_dev, non_blocking=True)
            st.synchronize()
            host = self._summ_host.numpy().copy()
        rows = host[:n_hist].reshape(len(tags), self._HROW)
        stats = {t: (r[0], r[1], r[2], r[3], r[4], r[5:]) for t, r in zip(tags, rows)}
        bad = host[n_hist:n_hist + n_bad].view(np.int32)[:len(tags)]
        l = self._loss_dict(host[n_hist + n_bad:].view(np.float32))
        return l, stats, [t for t, f in zip(tags, bad) if f]

    def histograms(self, x, y_r, a) -> dict:
        """The histograms `log` writes, for rows x and targets y_r, a: {tag: (min, max, num, sum, sum_squares, counts)}, TF's
        histogram::Histogram with its 1551 default buckets (ga3c_b200.summaries.LIMITS), computed on the GPU.  The tags
        (`_hist_tags`): weights_<variable name> (tf.summary's tag cleaning, e.g. weights_dense1/w_0) for every variable in TF
        creation order, then the activations of the hidden layers, activation_v and activation_p (see the subclass's `log`).
        Raises ValueError on a NaN / Inf."""
        _, stats, bad = self._summaries(x, y_r, a)
        if bad:
            raise self._nonfinite(bad)
        return stats

    # ------------------------------------------------------------------ introspection (tests / profiling)
    def launch_count(self) -> int:
        return int(getattr(self._lib, self._PREFIX + "launch_count")(self._h))

    def kernel_timing(self, max_records: int):
        """Bracket every kernel of the path with CUDA events on its launch stream (0 = off)."""
        self._call("timing_enable", int(max_records))

    def kernel_times(self) -> dict:
        """{kernel name: (total ms, launches)} of the kernels launched since the last call; synchronises the device."""
        n = self._lib.ga3c_kernel_count()
        tot, cnt = (C.c_double * n)(), (C.c_int64 * n)()
        self._call("timing_collect", tot, cnt, n)
        return {self._lib.ga3c_kernel_name(k).decode(): (tot[k], cnt[k]) for k in range(n) if cnt[k]}

    # ------------------------------------------------------------------ reference accessors
    # ------------------------------------------------------------------ reference accessors
    def predict_single(self, x):            # NetworkVP.py:237-238
        return self.predict_p(x[None, :])[0]

    def predict_v(self, x):                 # NetworkVP.py:240-242
        return self.predict_p_and_v(x)[1]

    def predict_p(self, x):                 # NetworkVP.py:244-246
        return self.predict_p_and_v(x)[0]

    def get_variables_names(self):          # NetworkVP.py:284-285 (TF creation order; gradient-less variables included)
        return list(self._table.keys())

    def get_variable_value(self, name):     # NetworkVP.py:287-288
        o, s = self._table[name]
        return self._download(0)[o:o + int(np.prod(s))].reshape(s).copy()

    def log(self, x, y_r, a, training_step, feed_dict=None):
        """NetworkVP.py:259-265 writes TensorBoard summaries from a second forward pass.  Here the same
        scalars (Pcost_advantage, Pcost_entropy, Pcost, Vcost, LearningRate, Beta) are appended to
        logs/<model_name>/scalars.csv."""
        self._log_csv(self.losses(x, y_r, a), training_step)

    def _log_csv(self, l: dict, training_step):
        os.makedirs(os.path.join("logs", self.model_name), exist_ok=True)
        with open(os.path.join("logs", self.model_name, "scalars.csv"), "a") as f:
            f.write(f"{training_step},{l['cost_p_1']},{l['cost_p_2']},{l['cost_p']},{l['cost_v']},"
                    f"{self.learning_rate},{self.beta}\n")

    @staticmethod
    def _nonfinite(tags):
        # HistogramSummary's InvalidArgument: "Nan in summary histogram for: <tag>" (or "Infinity ...")
        return ValueError("NaN or Infinity in summary histogram for: " + ", ".join(tags))

    def _log_summaries(self, l: dict, stats: dict, bad: list, training_step):
        """`log` of a network with TensorBoard histograms: the CSV line, then ValueError if a histogram holds a NaN / Inf (no
        event written), else the six scalars and `stats` at step training_step in the event file of logs/<model_name>."""
        self._log_csv(l, training_step)
        if bad:
            raise self._nonfinite(bad)
        if getattr(self, "_events", None) is None:
            self._events = summaries.EventLog(os.path.join("logs", self.model_name))
        values = (l["cost_p_1"], l["cost_p_2"], l["cost_p"], l["cost_v"], self.learning_rate, self.beta)
        self._events.write(int(training_step), dict(zip(summaries.SCALAR_TAGS, values)), stats)

    # ------------------------------------------------------------------ the arena as named tensors
    def _split(self, arena: np.ndarray):
        return {k: arena[o:o + int(np.prod(s))].reshape(s).copy() for k, (o, s) in self._table.items()}

    def _join(self, which: int, tensors: dict) -> np.ndarray:
        arena = self._download(which)
        for k, v in tensors.items():
            o, s = self._table[k]
            v = np.asarray(v, dtype=np.float32)
            if v.shape != tuple(s):
                raise ValueError(f"{k}: expected shape {s}, got {v.shape}")
            arena[o:o + v.size] = v.ravel()
        return arena

    def get_variables(self):
        return self._split(self._download(0))

    def set_variables(self, tensors: dict):
        self._upload(0, self._join(0, tensors))

    def get_slots(self, optimizer: int = 0):
        """(ms, mom) of the RMSProp optimizer; with Config.DUAL_RMSPROP optimizer 0 minimises cost_p and 1 cost_v."""
        base = 2 if optimizer == 0 else 5
        return self._split(self._download(base)), self._split(self._download(base + 1))

    def set_slots(self, ms: dict = None, mom: dict = None, optimizer: int = 0):
        base = 2 if optimizer == 0 else 5
        if ms is not None:
            self._upload(base, self._join(base, ms))
        if mom is not None:
            self._upload(base + 1, self._join(base + 1, mom))

    # ------------------------------------------------------------------ checkpoints
    def _checkpoint_filename(self, episode):    # NetworkVP.py:267-268
        return 'checkpoints/%s_%08d' % (self.model_name, episode)

    def _get_episode_from_filename(self, filename):     # NetworkVP.py:270-272
        return int(re.split(r'/|_|\.', filename)[2])

    def save(self, episode):
        """NetworkVP.py:274-275: all global variables (weights, RMSProp slots, step), keyed by TF name."""
        fn = self._checkpoint_filename(episode) + ".npz"
        os.makedirs(os.path.dirname(fn), exist_ok=True)
        ms, mom = self.get_slots()
        blob = dict(self.get_variables())
        blob.update({k.replace(":0", "/RMSProp:0"): v for k, v in ms.items()})
        blob.update({k.replace(":0", "/RMSProp_1:0"): v for k, v in mom.items()})
        if self._dual:
            ms2, mom2 = self.get_slots(1)
            blob.update({k.replace(":0", "/RMSProp_2:0"): v for k, v in ms2.items()})
            blob.update({k.replace(":0", "/RMSProp_3:0"): v for k, v in mom2.items()})
        blob["step:0"] = np.array(self.get_global_step(), dtype=np.int64)
        np.savez(fn, **blob)
        return fn

    def load(self):
        """NetworkVP.py:277-282: latest checkpoint, or Config.LOAD_EPISODE; returns the episode number."""
        d = os.path.dirname(self._checkpoint_filename(episode=0))
        if getattr(self.config, "LOAD_EPISODE", 0) > 0:
            filename = self._checkpoint_filename(self.config.LOAD_EPISODE)
        else:
            cands = sorted(f for f in os.listdir(d) if f.startswith(self.model_name + "_") and f.endswith(".npz"))
            filename = os.path.join(d, cands[-1][:-4])
        z = np.load(filename + ".npz")
        names = self.get_variables_names()
        self.set_variables({k: z[k] for k in names})
        self.set_slots({k: z[k.replace(":0", "/RMSProp:0")] for k in names},
                       {k: z[k.replace(":0", "/RMSProp_1:0")] for k in names})
        if self._dual and names[0].replace(":0", "/RMSProp_2:0") in z:
            self.set_slots({k: z[k.replace(":0", "/RMSProp_2:0")] for k in names},
                           {k: z[k.replace(":0", "/RMSProp_3:0")] for k in names}, optimizer=1)
        self._set_global_step(int(z["step:0"]))
        self._after_load()
        return self._get_episode_from_filename(filename)

    def _after_load(self):
        """Hook: what a subclass does once a checkpoint is in place (data parallel: make the replicas agree)."""
