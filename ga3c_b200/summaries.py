"""TensorBoard summaries of `Network.log` (NetworkVP.py:152-173, :259-265): the six scalars and the weight / activation
histograms, written to an event file under logs/<model_name> as the reference's `tf.summary.FileWriter` does.

The histogram statistics come from the device (ga3c_histograms, ga3c_mlp_histograms); this module only turns them into TF's histogram encoding and
writes them with `torch.utils.tensorboard.SummaryWriter`, which needs the optional `tensorboard` package.
"""
from __future__ import annotations

import re
import sys
import warnings

import numpy as np

BUCKETS = 1551          # GA3C_HISTO_BUCKETS
ACTIVATION_TAGS = ("activation_n1", "activation_n2", "activation_d2", "activation_v", "activation_p")
SCALAR_TAGS = ("Pcost_advantage", "Pcost_entropy", "Pcost", "Vcost", "LearningRate", "Beta")


def default_limits() -> np.ndarray:
    """TF's default bucket limits (histogram.cc InitDefaultBuckets): 1e-12 * 1.1^k by repeated fp64 multiplication while
    below 1e20, then DBL_MAX, mirrored around 0.0."""
    pos, v = [], 1e-12
    while v < 1e20:
        pos.append(v)
        v *= 1.1
    pos.append(sys.float_info.max)
    return np.array([-p for p in reversed(pos)] + [0.0] + pos, dtype=np.float64)


LIMITS = default_limits()
assert LIMITS.size == BUCKETS


def clean_tag(name: str) -> str:
    """tf.summary's _clean_tag: every character outside [-/\\w.] becomes '_'."""
    return re.sub(r"[^-/\w\.]", "_", name)


def histogram_tags(variable_names, activation_tags=ACTIVATION_TAGS) -> list:
    """The histogram tags in the order of ga3c_histograms' sources: weights_<var.name> per variable, then the activations,
    by default the conv net's as upstream NetworkVP._create_tensor_board names them (n1, n2, d1, logits_v, softmax_p)."""
    return [clean_tag("weights_" + n) for n in variable_names] + list(activation_tags)


def mlp_histogram_tags(variables) -> list:
    """The histogram tags of an MLP network in the order of ga3c_mlp_histograms' sources.  variables: (TF name, live) pairs in
    creation order (ga3c_mlp_param_info).  weights_<var.name> for every variable, the gradient-less ones included; then
    activation_<layer scope> for every live hidden layer in forward order (the scope of a live variable outside the heads
    logits_v / logits_p: dense11_p ... dense1 for the fork NetworkVP, dense1_<n>_p for NetworkVP_discrate); then activation_v
    (logits_v) and activation_p (softmax_p; for the fork NetworkVP the atan2 output it aliases)."""
    names = [n for n, _ in variables]
    scopes = dict.fromkeys(n.split("/")[0] for n, live in variables if live and not n.startswith("logits_"))
    return histogram_tags(names, [clean_tag("activation_" + s) for s in scopes] + ["activation_v", "activation_p"])


def collapse(counts):
    """HistogramProto buckets as Histogram::EncodeToProto(preserve_zero_buckets=false) writes them: a run of empty buckets
    becomes one entry with the limit of the run's last bucket and a count of 0.  Returns (bucket_limit, bucket)."""
    counts = np.asarray(counts, dtype=np.float64)
    full = counts > 0.0
    keep = full.copy()
    keep[:-1] |= full[1:]            # the last bucket of an empty run: the next one is full ...
    keep[-1] = True                  # ... or there is none
    return LIMITS[keep].tolist(), counts[keep].tolist()


class EventLog:
    """An event file in `logdir`, created at the first write and flushed after every write.  Without the `tensorboard`
    package nothing is written and one warning is issued."""

    def __init__(self, logdir: str):
        self.logdir = logdir
        self._writer = None
        self._missing = False

    def write(self, step: int, scalars: dict, histograms: dict) -> bool:
        """scalars: {tag: value}; histograms: {tag: (min, max, num, sum, sum_squares, counts[1551])}.  True if written."""
        if self._writer is None and not self._missing:
            try:
                from torch.utils.tensorboard import SummaryWriter
            except ImportError as e:
                self._missing = True
                warnings.warn(f"Network.log writes logs/<model_name>/scalars.csv only: no TensorBoard event file without the "
                              f"tensorboard package ({e})", RuntimeWarning, stacklevel=4)   # the caller of log()
            else:
                self._writer = SummaryWriter(self.logdir)
        if self._writer is None:
            return False
        for tag, value in scalars.items():
            self._writer.add_scalar(tag, float(value), global_step=step)
        for tag, (mn, mx, num, s, ss, counts) in histograms.items():
            limits, buckets = collapse(counts)
            self._writer.add_histogram_raw(tag, min=float(mn), max=float(mx), num=float(num), sum=float(s),
                                           sum_squares=float(ss), bucket_limits=limits, bucket_counts=buckets,
                                           global_step=step)
        self._writer.flush()
        return True

    def close(self):
        if self._writer is not None:
            self._writer.close()
            self._writer = None
