"""CPU tests of the TensorBoard summaries of Network.log: the oracle's restatement of TF's histogram::Histogram (bucket limits,
upper_bound placement, the collapse of empty runs, tag cleaning), the product's copy of the limits and of the encoding, and the
event-writing half fed fixed statistics and read back with tensorboard's EventAccumulator."""
import os
import sys

import numpy as np
import pytest

from oracle import histogram_np as oh

DBL_MAX = sys.float_info.max


def test_default_limits():
    L = oh.LIMITS
    assert L.size == 1551 and L.dtype == np.float64
    assert L[775] == 0.0 and L[0] == -DBL_MAX and L[-1] == DBL_MAX
    assert np.array_equal(L, -L[::-1])                         # symmetric
    assert np.all(np.diff(L) > 0)
    assert L[776] == 1e-12 and L[-2] < 1e20 <= L[-2] * 1.1
    from ga3c_b200 import summaries
    assert np.array_equal(summaries.LIMITS, L) and summaries.BUCKETS == L.size


def test_upper_bound_placement():
    L = oh.LIMITS

    def bucket(x):
        return int(np.argmax(oh.histogram([x])[5]))

    for i in (1, 100, 700, 774, 776, 777, 900, 1549):
        assert bucket(L[i]) == i + 1                            # on a limit: the NEXT bucket
        assert bucket(np.nextafter(L[i], -np.inf)) == i
        assert bucket(np.nextafter(L[i], np.inf)) == i + 1
    assert bucket(0.0) == 776 and bucket(-0.0) == 776           # -0.0 == 0.0 for upper_bound
    assert bucket(5e-13) == 776 and bucket(-5e-13) == 775       # |x| < 1e-12
    assert bucket(1e-300) == 776 and bucket(-1e-300) == 775
    assert bucket(1e21) == 1550 and bucket(-1e21) == 1          # beyond the last finite limit
    mn, mx, num, s, ss, counts = oh.histogram(np.array([1.0, -2.0, 0.0, 3.0], np.float32))
    assert (mn, mx, num, s, ss) == (-2.0, 3.0, 4.0, 2.0, 14.0) and counts.sum() == 4
    mn, mx, num, s, ss, counts = oh.histogram(np.zeros(0))
    assert (mn, mx, num) == (DBL_MAX, -DBL_MAX, 0.0)
    with pytest.raises(oh.NonFiniteError, match="Nan in summary histogram for: t"):
        oh.histogram([1.0, np.nan], "t")
    with pytest.raises(oh.NonFiniteError, match="Infinity in summary histogram for: u"):
        oh.histogram([np.inf], "u")


def test_collapse_of_empty_runs():
    from ga3c_b200 import summaries
    L = oh.LIMITS
    counts = np.zeros(1551)
    counts[3] = 2.0
    counts[4] = 1.0
    counts[776] = 5.0
    want_limits = [L[2], L[3], L[4], L[775], L[776], L[1550]]
    want_counts = [0.0, 2.0, 1.0, 0.0, 5.0, 0.0]
    for enc in (oh.encode, summaries.collapse):
        lim, cnt = enc(counts)
        assert lim == want_limits and cnt == want_counts
        assert enc(np.zeros(1551)) == ([DBL_MAX], [0.0])        # one empty run: the last limit
        full = np.ones(1551)
        assert enc(full) == (list(L), list(full))
    c = np.zeros(1551)
    c[0] = 1.0
    assert oh.encode(c) == ([L[0], L[1550]], [1.0, 0.0]) == summaries.collapse(c)


def test_tag_cleaning():
    from ga3c_b200 import summaries
    for clean in (oh.clean_tag, summaries.clean_tag):
        assert clean("weights_dense1/w:0") == "weights_dense1/w_0"
        assert clean("weights_conv11/w:0") == "weights_conv11/w_0"
        assert clean("a b+c-d.e/f_g") == "a_b_c-d.e/f_g"
    names = list(__import__("oracle.oracle_np", fromlist=["PARAM_NAMES"]).PARAM_NAMES)
    tags = summaries.histogram_tags(names)
    assert len(tags) == 15 and tags[0] == "weights_conv11/w_0" and tags[9] == "weights_logits_p/b_0"
    assert tags[10:] == [t for t, _ in oh.ACTIVATIONS]
    assert summaries.SCALAR_TAGS == oh.SCALAR_TAGS


def test_event_file_round_trip(tmp_path):
    """EventLog (what Network.log writes through) fed fixed statistics: every scalar and histogram reads back from the event
    file at the given step with min / max / num / sum / sum_squares and the collapsed limits / counts as written."""
    pytest.importorskip("tensorboard")
    from tensorboard.backend.event_processing import event_accumulator
    from ga3c_b200 import summaries
    from oracle import oracle_np as onp
    rng = np.random.default_rng(5)
    tags = summaries.histogram_tags(onp.PARAM_NAMES)
    hist = {t: oh.histogram(rng.standard_normal(50 + 10 * i) * 10.0 ** (i - 7), t) for i, t in enumerate(tags)}
    scalars = dict(zip(summaries.SCALAR_TAGS, (1.5, -0.25, -1.25, 3.0, 3e-4, 0.01)))
    log = summaries.EventLog(str(tmp_path))
    for step in (1000, 2000):
        assert log.write(step, scalars, hist)
    log.close()
    acc = event_accumulator.EventAccumulator(str(tmp_path), size_guidance={event_accumulator.HISTOGRAMS: 0,
                                                                           event_accumulator.SCALARS: 0})
    acc.Reload()
    assert sorted(acc.Tags()["scalars"]) == sorted(summaries.SCALAR_TAGS)
    assert sorted(acc.Tags()["histograms"]) == sorted(tags)
    for t, v in scalars.items():
        ev = acc.Scalars(t)
        assert [e.step for e in ev] == [1000, 2000] and all(np.float32(e.value) == np.float32(v) for e in ev)
    for t, (mn, mx, num, s, ss, counts) in hist.items():
        ev = acc.Histograms(t)
        assert [e.step for e in ev] == [1000, 2000]
        h = ev[-1].histogram_value
        lim, cnt = oh.encode(counts)
        assert (h.min, h.max, h.num, h.sum, h.sum_squares) == (mn, mx, num, s, ss)
        assert list(h.bucket_limit) == lim and list(h.bucket) == cnt
