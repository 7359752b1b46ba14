"""GPU tests of the TensorBoard summaries: the histogram kernel (ga3c_debug_histogram) against the numpy restatement of TF's
histogram::Histogram (oracle/histogram_np.py) on crafted fp32 / bf16 inputs, Network.histograms against the oracle run over the
network's own variables and activations, and Network.log's event file."""
import numpy as np
import pytest

from oracle import histogram_np as oh
from oracle import oracle_np as onp
from _parity import ga3c  # noqa: F401  (pytest fixture)

pytestmark = pytest.mark.gpu

ROW = 5 + 1551


def device_histogram(t):
    """ga3c_debug_histogram over one flat fp32 / bf16 CUDA tensor: (row of 5 + 1551 doubles, non-finite flag)."""
    import torch
    from ga3c_b200 import _capi
    lib = _capi.load()
    out = torch.empty(ROW, dtype=torch.float64, device=t.device)
    bad = torch.empty(1, dtype=torch.int32, device=t.device)
    dtype = {torch.float32: 0, torch.bfloat16: 1}[t.dtype]
    _capi.check(lib.ga3c_debug_histogram(t.data_ptr(), dtype, t.numel(), out.data_ptr(), bad.data_ptr(), None),
                "ga3c_debug_histogram")
    torch.cuda.synchronize()
    return out.cpu().numpy(), int(bad.item())


def assert_matches(got, x, tag=""):
    """counts, min, max, num exactly; sum within 1e-12 * sum|x|, sum_squares within 1e-12 * sum x^2."""
    x = np.asarray(x, dtype=np.float64).ravel()
    mn, mx, num, s, ss, counts = oh.histogram(x, tag)
    got = np.asarray(got, dtype=np.float64)
    assert np.array_equal(got[5:], counts), (tag, np.nonzero(got[5:] != counts)[0][:10])
    assert (got[0], got[1], got[2]) == (mn, mx, num), (tag, got[:3], (mn, mx, num))
    assert abs(got[3] - s) <= 1e-12 * np.abs(x).sum(), (tag, got[3], s)
    assert abs(got[4] - ss) <= 1e-12 * (x * x).sum(), (tag, got[4], ss)


def crafted_values():
    """The float neighbours just below, at and just above every finite limit, zeros of both signs, magnitudes below 1e-12
    (denormals included), large magnitudes and negatives."""
    L = oh.LIMITS[1:-1]
    f = L.astype(np.float32)
    f = f[np.isfinite(f)]
    near = np.concatenate([np.nextafter(f, np.float32(-np.inf)), f, np.nextafter(f, np.float32(np.inf))])
    extra = np.array([0.0, -0.0, 1e-13, -1e-13, 9.99e-13, -9.99e-13, 1e-30, -1e-30, 1e-40, -1e-45, 1e20, -1e20, 1e25, -1e25,
                      3.4e38, -3.4e38, 1.0, -1.0, 0.5, -123.25], dtype=np.float32)
    return np.concatenate([near, extra]).astype(np.float32)


def test_kernel_crafted_fp32_and_bf16(ga3c):
    import torch
    x = crafted_values()
    rng = np.random.default_rng(0)
    x = x[rng.permutation(x.size)]
    for n in (x.size, 1, 3, 7, 13, 4101):                        # ragged tails, one chunk, one value
        t = torch.from_numpy(x[:n].copy()).cuda()
        got, bad = device_histogram(t)
        assert bad == 0
        assert_matches(got, x[:n], f"fp32 n={n}")
        tb = t.to(torch.bfloat16)
        tb = tb[torch.isfinite(tb)]                               # +-3.4e38 rounds to +-inf in bf16
        got, bad = device_histogram(tb)
        assert bad == 0
        assert_matches(got, tb.float().cpu().numpy(), f"bf16 n={n}")
    # the bf16 neighbours of every limit
    L = oh.LIMITS[1:-1]
    b = torch.from_numpy(L.astype(np.float32)).to(torch.bfloat16)
    bits = b.view(torch.int16)
    nb = torch.cat([b, (bits + 1).view(torch.bfloat16), (bits - 1).view(torch.bfloat16)])
    nb = nb[torch.isfinite(nb.float())].cuda()
    got, bad = device_histogram(nb)
    assert bad == 0
    assert_matches(got, nb.float().cpu().numpy(), "bf16 limits")


def test_kernel_relu_like_10m_deterministic(ga3c):
    import torch
    rng = np.random.default_rng(1)
    n = 10_000_003
    x = (rng.standard_normal(n) * np.exp(rng.uniform(-8, 4, n))).astype(np.float32)
    x[rng.random(n) < 0.5] = 0.0
    x = np.maximum(x, 0.0) - 0.01 * (rng.random(n) < 0.01) * np.abs(x)       # mostly ReLU output, a few negatives
    x = x.astype(np.float32)
    t = torch.from_numpy(x).cuda()
    for tt, ref in ((t, x), (t.to(torch.bfloat16), None)):
        ref = tt.float().cpu().numpy() if ref is None else ref
        got, bad = device_histogram(tt)
        assert bad == 0
        assert_matches(got, ref, str(tt.dtype))
        again, _ = device_histogram(tt)
        assert again.tobytes() == got.tobytes()                  # bit-identical across calls


def test_kernel_flags_nan_and_inf(ga3c):
    import torch
    from ga3c_b200 import _capi
    x = np.linspace(-1, 1, 1000, dtype=np.float32)
    for bad_value in (np.nan, np.inf, -np.inf):
        y = x.copy()
        y[517] = bad_value
        for dt in (torch.float32, torch.bfloat16):
            _, bad = device_histogram(torch.from_numpy(y).cuda().to(dt))
            assert bad != 0, (bad_value, dt)
    _, bad = device_histogram(torch.from_numpy(x).cuda())
    assert bad == 0
    t = torch.from_numpy(x).cuda()
    with pytest.raises(_capi.Ga3cError, match="aligned"):
        _capi.check(_capi.load().ga3c_debug_histogram(t.data_ptr() + 4, 0, 16, t.data_ptr(), t.data_ptr(), None), "x")


def _net(ga3c, b, seed=7):
    rng = np.random.default_rng(seed)
    params = onp.init_params(rng, 6)
    k = onp.synth_frames_u8(rng, b)
    x = onp.normalise(k)
    y_r, a = onp.synth_targets(rng, b)
    net = ga3c.Network("gpu:0", "histtest", 6, max_batch=max(b, 32))
    net.set_variables(params)
    return net, params, k, x, y_r, a


@pytest.mark.parametrize("b", [1, 37, 1024])
def test_network_histograms_match_the_oracle(ga3c, b):
    net, params, k, x, y_r, a = _net(ga3c, b)
    got = net.histograms(x, y_r, a)
    n1, n2, d1 = net.workspace(0), net.workspace(1), net.workspace(2)
    p, v = net.predict_p_and_v(x)
    values = {oh.clean_tag("weights_" + name): t for name, t in net.get_variables().items()}
    values.update(zip([t for t, _ in oh.ACTIVATIONS], (n1, n2, d1, v, p)))
    assert list(got) == list(values)
    for tag, vals in values.items():
        assert_matches(np.concatenate([np.array(got[tag][:5]), got[tag][5]]), vals, tag)
    # uint8 frames: bit-identical to their float32 frames
    got8 = net.histograms(k, y_r, a)
    for tag in got:
        assert all(np.array_equal(np.asarray(g), np.asarray(h)) for g, h in zip(got[tag], got8[tag])), tag


def test_log_writes_events_and_leaves_the_state_alone(ga3c, tmp_path, monkeypatch):
    pytest.importorskip("tensorboard")
    from tensorboard.backend.event_processing import event_accumulator
    from ga3c_b200 import summaries
    monkeypatch.chdir(tmp_path)
    net, params, k, x, y_r, a = _net(ga3c, 24)
    net.learning_rate, net.beta = 1e-4, 0.02
    ms0, mom0 = net.get_slots()
    l = net.losses(x, y_r, a)
    line = f"1000,{l['cost_p_1']},{l['cost_p_2']},{l['cost_p']},{l['cost_v']},{net.learning_rate},{net.beta}"
    net.log(x, y_r, a, 1000)
    assert open(tmp_path / "logs" / "histtest" / "scalars.csv").read() == line + "\n"
    w = net.get_variables()
    ms, mom = net.get_slots()
    assert all(np.array_equal(w[n], params[n]) and np.array_equal(ms[n], ms0[n]) and np.array_equal(mom[n], mom0[n]) for n in w)
    assert net.get_global_step() == 0
    hist = net.histograms(x, y_r, a)

    acc = event_accumulator.EventAccumulator(str(tmp_path / "logs" / "histtest"),
                                             size_guidance={event_accumulator.HISTOGRAMS: 0, event_accumulator.SCALARS: 0})
    acc.Reload()
    assert sorted(acc.Tags()["scalars"]) == sorted(summaries.SCALAR_TAGS)
    assert sorted(acc.Tags()["histograms"]) == sorted(hist) and len(hist) == 15
    for tag, value in zip(summaries.SCALAR_TAGS, (l["cost_p_1"], l["cost_p_2"], l["cost_p"], l["cost_v"], 1e-4, 0.02)):
        (e,) = acc.Scalars(tag)
        assert e.step == 1000 and np.float32(e.value) == np.float32(value), tag
    for tag, (mn, mx, num, s, ss, counts) in hist.items():
        (e,) = acc.Histograms(tag)
        h = e.histogram_value
        assert e.step == 1000 and (h.min, h.max, h.num, h.sum, h.sum_squares) == (mn, mx, num, s, ss), tag
        assert (list(h.bucket_limit), list(h.bucket)) == oh.encode(counts), tag

    # a NaN in dense1/b: the CSV line is written, then the error names the tag; no event for that call
    bad = dict(params)
    bad["dense1/b:0"] = params["dense1/b:0"].copy()
    bad["dense1/b:0"][3] = np.nan
    net.set_variables(bad)
    with pytest.raises(ValueError, match="weights_dense1/b_0"):
        net.log(x, y_r, a, 2000)
    rows = open(tmp_path / "logs" / "histtest" / "scalars.csv").read().splitlines()
    assert len(rows) == 2 and rows[1].startswith("2000,")
    acc.Reload()
    assert [e.step for e in acc.Histograms("weights_dense1/b_0")] == [1000]
