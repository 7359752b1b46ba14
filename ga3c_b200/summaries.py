"""TensorBoard summaries of `Network.log` (NetworkVP.py:152-173, :259-265): the six scalars and the weight / activation
histograms, written to an event file under logs/<model_name> as the reference's `tf.summary.FileWriter` does.

The histogram statistics come from the device (ga3c_histograms); this module only turns them into TF's histogram encoding and
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


def histogram_tags(variable_names) -> list:
    """The tags of the 15 histograms in the order of ga3c_histograms' sources: weights_<var.name> per variable, then the
    activations as upstream NetworkVP._create_tensor_board names them (n1, n2, d1, logits_v, softmax_p)."""
    return [clean_tag("weights_" + n) for n in variable_names] + list(ACTIVATION_TAGS)


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
                              f"tensorboard package ({e})", RuntimeWarning, stacklevel=3)
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
