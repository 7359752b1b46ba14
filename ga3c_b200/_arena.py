"""What the conv `Network` and the low-dimensional MLP networks share on the host side: the reference's small accessors, the
flat parameter arena seen as a dict of TF-named tensors, RMSProp slots, checkpoints, the scalar log and the writing of
`log`'s TensorBoard event file.

A subclass provides `_table` ({TF variable name: (offset, shape)} into the fp32 arena, in TF creation order), `_download(which)`
/ `_upload(which, arena)` (arena ids: 0 weights, 1 gradients, 2 / 3 ms / mom of the first optimizer, 5 / 6 of the second),
`get_global_step()`, `_set_global_step(step)`, `losses(x, y_r, a)`, and the attributes `model_name`, `config`, `_dual`,
`learning_rate`, `beta`.
"""
from __future__ import annotations

import os
import re

import numpy as np

from . import summaries


class ArenaNetworkMixin:
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
