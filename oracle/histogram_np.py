"""numpy restatement of TensorFlow's histogram::Histogram and the histogram summaries of NetworkVP._create_tensor_board.
TEST INFRASTRUCTURE ONLY.

TensorFlow is not available to this repository, so every point tagged [TF-SEMANTICS] below is a restatement of TF 1.x
behaviour (tensorflow/core/lib/histogram/histogram.cc, tensorflow/core/kernels/summary_op.cc, tensorflow/python/ops/
summary_op_util.py) that is not checked against TF itself.
"""
from __future__ import annotations

import re
import sys

import numpy as np

DBL_MAX = sys.float_info.max


def default_limits() -> np.ndarray:
    """[TF-SEMANTICS] Histogram::InitDefaultBuckets: positive limits 1e-12, *1.1, ... while < 1e20 (fp64, repeated
    multiplication), then DBL_MAX; the full table is -reversed(pos), 0.0, pos: 1551 limits with 0.0 at index 775."""
    pos = []
    v = 1e-12
    while v < 1e20:
        pos.append(v)
        v *= 1.1
    pos = pos + [DBL_MAX]
    return np.array([-p for p in reversed(pos)] + [0.0] + pos, dtype=np.float64)


LIMITS = default_limits()


class NonFiniteError(ValueError):
    """[TF-SEMANTICS] HistogramSummary fails with InvalidArgument on a NaN ("Nan in summary histogram for: <tag>") or an Inf
    ("Infinity in summary histogram for: <tag>")."""


def histogram(values, tag: str = "") -> tuple:
    """[TF-SEMANTICS] Histogram::Add for every value: x as a double, bucket = std::upper_bound(limits, x) (a value equal to a
    limit goes into the NEXT bucket), min / max start at +-DBL_MAX, num / sum / sum_squares accumulate in double.
    Returns (min, max, num, sum, sum_squares, counts[1551])."""
    x = np.asarray(values).astype(np.float64).ravel()
    if np.isnan(x).any():
        raise NonFiniteError(f"Nan in summary histogram for: {tag}")
    if np.isinf(x).any():
        raise NonFiniteError(f"Infinity in summary histogram for: {tag}")
    idx = np.searchsorted(LIMITS, x, side="right")
    counts = np.bincount(idx, minlength=LIMITS.size).astype(np.float64)[:LIMITS.size]
    mn = min(DBL_MAX, x.min()) if x.size else DBL_MAX
    mx = max(-DBL_MAX, x.max()) if x.size else -DBL_MAX
    return mn, mx, float(x.size), float(x.sum()), float((x * x).sum()), counts


def encode(counts) -> tuple:
    """[TF-SEMANTICS] Histogram::EncodeToProto(proto, preserve_zero_buckets=false): a run of empty buckets collapses into one
    entry that carries the limit of the run's LAST bucket and a count of 0; an empty result becomes (DBL_MAX, 0).
    Returns (bucket_limit, bucket) lists."""
    limits, buckets = [], []
    i = 0
    while i < len(counts):
        end, c = LIMITS[i], counts[i]
        i += 1
        if c <= 0.0:
            while i < len(counts) and counts[i] <= 0.0:
                end, c = LIMITS[i], counts[i]
                i += 1
        limits.append(float(end))
        buckets.append(float(c))
    if not limits:
        return [DBL_MAX], [0.0]
    return limits, buckets


def clean_tag(name: str) -> str:
    """[TF-SEMANTICS] summary_op_util._clean_tag: characters outside [-/\\w.] become '_' (weights_conv11/w:0 ->
    weights_conv11/w_0)."""
    return re.sub(r"[^-/\w\.]", "_", name)


# [TF-SEMANTICS] upstream NVlabs NetworkVP._create_tensor_board: the six scalars, one histogram per trainable variable
# ("weights_%s" % var.name, TF creation order) and these activations
SCALAR_TAGS = ("Pcost_advantage", "Pcost_entropy", "Pcost", "Vcost", "LearningRate", "Beta")
ACTIVATIONS = (("activation_n1", "n1"), ("activation_n2", "n2"), ("activation_d2", "d1"), ("activation_v", "logits_v"),
               ("activation_p", "softmax_p"))

