"""GPU tests of the MLP networks' TensorBoard summaries: _MlpNetwork.histograms against the numpy restatement of TF's
histogram::Histogram (oracle/histogram_np.py) run over the network's own variables, layer outputs and predictions, on the
fp32 FMA path and the tensor-core path; bit-identical reruns; log's CSV line and event file; the batch check of
ga3c_mlp_histograms."""
import numpy as np
import pytest

from oracle import histogram_np as oh
from oracle import oracle_mlp as om
from _parity import make_mlp_case, make_mlp_net

pytestmark = pytest.mark.gpu

CASES = [("fork_vp", 3, 1), ("fork_vp", 4, 2), ("discrate", 4, 2)]


@pytest.fixture(scope="module")
def mlp():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; there is no CPU fallback")
    from ga3c_b200 import mlp_network
    return mlp_network


def assert_matches(got, x, tag=""):
    """counts, min, max, num exactly; sum within 1e-12 * sum|x|, sum_squares within 1e-12 * sum x^2."""
    mn, mx, num, s, ss, counts = got
    x = np.asarray(x, dtype=np.float64).ravel()
    r_mn, r_mx, r_num, r_s, r_ss, r_counts = oh.histogram(x, tag)
    assert np.array_equal(counts, r_counts), (tag, np.nonzero(counts != r_counts)[0][:10])
    assert (mn, mx, num) == (r_mn, r_mx, r_num), (tag, (mn, mx, num), (r_mn, r_mx, r_num))
    assert abs(s - r_s) <= 1e-12 * np.abs(x).sum(), (tag, s, r_s)
    assert abs(ss - r_ss) <= 1e-12 * (x * x).sum(), (tag, ss, r_ss)


def check_against_the_network(net, kind, x, y_r, act, dense_layers=om.DISCRATE_DENSE_LAYERS, variables=None):
    """histograms(), then the values they describe read back from the network: the variables (or `variables`), the layer
    outputs of the forward it just ran (before any further predict can rewrite them), p and v."""
    b = x.shape[0]
    got = net.histograms(x, y_r, act)
    layers = om.layers_of(kind, dense_layers)
    acts = [net.workspace(0, l, b) for l in range(len(layers))]
    p, v = net.predict_p_and_v(x)
    w = net.get_variables() if variables is None else variables
    values = {oh.clean_tag("weights_" + n): w[n] for n in net.get_variables_names()}
    values.update(("activation_" + name, t) for (name, _, _), t in zip(layers, acts))
    values.update(activation_v=v, activation_p=p)
    assert list(got) == list(values)
    for tag, vals in values.items():
        assert_matches(got[tag], vals, tag)
    return got


@pytest.mark.parametrize("kind,s,a", CASES)
@pytest.mark.parametrize("b", [1, 63, 1000, 4097])
def test_histograms_match_the_oracle(mlp, kind, s, a, b):
    params, x, y_r, act = make_mlp_case(kind, s, a, b)
    net = make_mlp_net(mlp, kind, s, a, max_batch=b)
    net.set_variables(params)
    check_against_the_network(net, kind, x, y_r, act)


@pytest.mark.parametrize("s,a", [(3, 1), (8, 2)])
def test_histograms_on_the_tensor_core_path(mlp, monkeypatch, s, a):
    """GA3C_MLP_TC=1: the wide layers of the fork NetworkVP as tcgen05 GEMMs from one row on, the narrow ends as streaming
    kernels (one action, state_dim <= 4; predict then also writes the layer workspace) or as the fused kernel's phases."""
    monkeypatch.setenv("GA3C_MLP_TC", "1")
    kind, b = "fork_vp", 1000
    params, x, y_r, act = make_mlp_case(kind, s, a, b, seed=3)
    net = make_mlp_net(mlp, kind, s, a, max_batch=b)
    net.set_variables(params)
    n0 = net.launch_count()
    net.predict_p_and_v(x)
    assert net.launch_count() - n0 == (5 if a == 1 and s <= 4 else 1)      # the path the shape selects
    check_against_the_network(net, kind, x, y_r, act)


def test_discrate_with_eight_dense_layers_uses_every_source(mlp):
    """Config.DENSE_LAYERS with 8 entries: 20 variables + 1 live layer + v + p = 23 sources.  After training steps the
    gradient-less layers still hold their initial values, and their histograms say so."""
    dense = (10, 20, 30, 40, 50, 60, 70, 16)

    class Cfg(mlp._DefaultConfig):
        DENSE_LAYERS = dense
    kind, s, a, b = "discrate", 4, 2, 777
    params, x, y_r, act = make_mlp_case(kind, s, a, b, seed=5, dense_layers=dense)
    net = make_mlp_net(mlp, kind, s, a, config=Cfg, max_batch=b)
    net.set_variables(params)
    assert net._lib.ga3c_mlp_histogram_count(net._h) == 23
    for _ in range(3):
        net.train(x, y_r, act, None, None, 0)
    trained = net.get_variables()
    assert not np.array_equal(trained["logits_v/w:0"], params["logits_v/w:0"])
    got = check_against_the_network(net, kind, x, y_r, act, dense_layers=dense)
    assert len(got) == 23
    for n in om.dead_params(kind, dense):
        assert_matches(got[oh.clean_tag("weights_" + n)], params[n], n)


def test_histograms_are_bit_identical_from_call_to_call(mlp):
    kind, s, a, b = "fork_vp", 3, 1, 65536           # multi-block sources: the fp64 moments are merged in block order
    params, x, y_r, act = make_mlp_case(kind, s, a, b, seed=9)
    net = make_mlp_net(mlp, kind, s, a, max_batch=b)
    net.set_variables(params)
    first = net.histograms(x, y_r, act)
    again = net.histograms(x, y_r, act)
    assert list(first) == list(again)
    for tag in first:
        assert all(np.asarray(u).tobytes() == np.asarray(w).tobytes() for u, w in zip(first[tag], again[tag])), tag


def test_kernel_times_report_the_histograms(mlp):
    kind, s, a, b = "discrate", 4, 2, 100
    params, x, y_r, act = make_mlp_case(kind, s, a, b)
    net = make_mlp_net(mlp, kind, s, a)
    net.set_variables(params)
    net.kernel_timing(64)
    net.kernel_times()
    net.histograms(x, y_r, act)
    kt = net.kernel_times()
    net.kernel_timing(0)
    assert kt["histograms"][1] == 2                  # histo_kernel + histo_merge_kernel


@pytest.mark.parametrize("kind,s,a", [("fork_vp", 3, 1), ("discrate", 4, 2)])
def test_log_writes_events_and_leaves_the_state_alone(mlp, tmp_path, monkeypatch, kind, s, a):
    pytest.importorskip("tensorboard")
    from tensorboard.backend.event_processing import event_accumulator
    from ga3c_b200 import summaries
    monkeypatch.chdir(tmp_path)
    params, x, y_r, act = make_mlp_case(kind, s, a, 300, seed=17)
    net = make_mlp_net(mlp, kind, s, a)
    net.set_variables(params)
    net.learning_rate, net.beta = 1e-4, 0.02
    ms0, mom0 = net.get_slots()
    l = net.losses(x, y_r, act)
    line = f"1000,{l['cost_p_1']},{l['cost_p_2']},{l['cost_p']},{l['cost_v']},{net.learning_rate},{net.beta}"
    net.log(x, y_r, act, 1000)
    logdir = tmp_path / "logs" / net.model_name
    assert open(logdir / "scalars.csv").read() == line + "\n"
    w = net.get_variables()
    ms, mom = net.get_slots()
    assert all(np.array_equal(w[n], params[n]) and np.array_equal(ms[n], ms0[n]) and np.array_equal(mom[n], mom0[n]) for n in w)
    assert net.get_global_step() == 0
    hist = net.histograms(x, y_r, act)

    acc = event_accumulator.EventAccumulator(str(logdir), size_guidance={event_accumulator.HISTOGRAMS: 0,
                                                                         event_accumulator.SCALARS: 0})
    acc.Reload()
    assert sorted(acc.Tags()["scalars"]) == sorted(summaries.SCALAR_TAGS)
    assert sorted(acc.Tags()["histograms"]) == sorted(hist)
    for tag, value in zip(summaries.SCALAR_TAGS, (l["cost_p_1"], l["cost_p_2"], l["cost_p"], l["cost_v"], 1e-4, 0.02)):
        (e,) = acc.Scalars(tag)
        assert e.step == 1000 and np.float32(e.value) == np.float32(value), tag
    for tag, (mn, mx, num, s_, ss, counts) in hist.items():
        (e,) = acc.Histograms(tag)
        h = e.histogram_value
        assert e.step == 1000 and (h.min, h.max, h.num, h.sum, h.sum_squares) == (mn, mx, num, s_, ss), tag
        assert (list(h.bucket_limit), list(h.bucket)) == oh.encode(counts), tag

    # a NaN in logits_v/b: the CSV line is written, then the error names the tag; no event for that call
    bad = dict(params)
    bad["logits_v/b:0"] = np.array([np.nan], np.float32)
    net.set_variables(bad)
    with pytest.raises(ValueError, match="weights_logits_v/b_0"):
        net.log(x, y_r, act, 2000)
    rows = open(logdir / "scalars.csv").read().splitlines()
    assert len(rows) == 2 and rows[1].startswith("2000,")
    acc.Reload()
    assert [e.step for e in acc.Histograms("weights_logits_v/b_0")] == [1000]
    assert [e.step for e in acc.Scalars("Vcost")] == [1000]


def test_histograms_refuse_a_batch_other_than_the_last_forward(mlp):
    import torch
    from ga3c_b200 import _capi
    kind, s, a = "fork_vp", 3, 1
    params, x, y_r, act = make_mlp_case(kind, s, a, 64)
    net = make_mlp_net(mlp, kind, s, a)
    net.set_variables(params)
    lib, n_src = net._lib, net._lib.ga3c_mlp_histogram_count(net._h)
    out = torch.empty(n_src * (5 + 1551), dtype=torch.float64, device="cuda:0")
    bad = torch.empty(n_src, dtype=torch.int32, device="cuda:0")
    p = torch.zeros(64, a, device="cuda:0")
    v = torch.zeros(64, device="cuda:0")

    def call(b):
        return lib.ga3c_mlp_histograms(net._h, b, p.data_ptr(), v.data_ptr(), out.data_ptr(), bad.data_ptr(), None)

    assert call(16) != 0                                     # no forward yet on this handle
    assert "batch differs" in lib.ga3c_last_error().decode()
    net.losses(x[:32], y_r[:32], act[:32])                   # forward of 32 rows
    net.predict_p_and_v(x)                                   # fused predict of 64 rows: the layer workspace holds 32 rows
    assert call(64) != 0 and "batch differs" in lib.ga3c_last_error().decode()
    assert call(16) != 0
    assert call(32) == 0
    torch.cuda.synchronize()
    net._ensure(4096)                                        # a new workspace holds no rows
    assert call(32) != 0
    with pytest.raises(_capi.Ga3cError):
        _capi.check(lib.ga3c_mlp_histograms(net._h, 32, 0, v.data_ptr(), out.data_ptr(), bad.data_ptr(), None), "null p")
