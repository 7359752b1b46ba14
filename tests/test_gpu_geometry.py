"""GPU tests (`-m gpu`) of the conv network at input geometries other than 84x84x4 (Config.IMAGE_HEIGHT, IMAGE_WIDTH,
STACKED_FRAMES), which run the generic trunk (conv_gen.cu), against the geometry-parameterised bf16 oracle
(tests/_geometry_oracle.py) with the tolerances of test_gpu_parity.py."""
import numpy as np
import pytest

from oracle import oracle_np as onp
from oracle import histogram_np as hnp
import _geometry_oracle as go
from _parity import err

pytestmark = pytest.mark.gpu

TOL_P, TOL_V = 2e-5, 2e-4
TOL_ACT_REL = 2.0 ** -7
TOL_LOSS_REL = 1e-4
TOL_GRAD_REL = 2e-3
TOL_W_ABS = 2e-6

GEOMETRIES = [(84, 84, 1), (84, 84, 3), (42, 42, 4), (105, 80, 4), (100, 100, 2), (8, 8, 1), (128, 128, 4)]
IDS = [f"{h}x{w}x{c}" for h, w, c in GEOMETRIES]
GEN_KERNELS = {"gen_wprep", "gen_im2col11", "gen_conv11", "gen_im2col12", "gen_conv12", "gen_conv12_dgrad", "gen_col2im",
               "gen_conv12_wgrad", "gen_conv11_wgrad"}


@pytest.fixture(scope="module")
def ga3c():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; there is no CPU fallback")
    import ga3c_b200
    return ga3c_b200


def config(hwc, **kw):
    from ga3c_b200 import Config

    class Cfg(Config):
        pass
    Cfg.IMAGE_HEIGHT, Cfg.IMAGE_WIDTH, Cfg.STACKED_FRAMES = hwc
    for k, v in kw.items():
        setattr(Cfg, k, v)
    return Cfg


def make_net(ga3c, hwc, max_batch, num_actions=6, **kw):
    return ga3c.Network("gpu:0", "geo", num_actions, hwc[0] * hwc[1] * hwc[2], config=config(hwc, **kw), max_batch=max_batch)


def case(g, b, seed=12345, num_actions=6):
    rng = np.random.default_rng(seed)
    params = go.init_params(rng, g, num_actions)
    k = go.synth_frames_u8(rng, g, b)
    y_r, a = onp.synth_targets(rng, b, num_actions)
    return params, k, go.normalise(k), y_r, a


def layer_report(net, g, params, x, y_r, a, **kw):
    net.set_variables(params)
    p, v = net.predict_p_and_v(x)
    losses_ref, grads_ref, f = go.loss_and_grads(g, params, x, y_r, a, quant="bf16", keep=True, **kw)
    rep = {"p": err(p, f["p"]), "v": err(v, f["v"])}
    losses = net.losses(x, y_r, a)
    b = x.shape[0]
    ws = {i: net.workspace(i) for i in (0, 1, 2, 3, 4, 5)}
    rep["n1"] = err(ws[0], f["n1"].reshape(b, -1))
    rep["n2"] = err(ws[1], f["n2"].reshape(b, -1))
    rep["d1"] = err(ws[2], f["d1"])
    rep["dd1"] = err(ws[3], f["dd1"])
    # layer-local data gradients: the oracle's arithmetic on the CUDA path's own stored inputs (see tests/_parity.py)
    n1_mask, n2_mask = ws[0].reshape(b, -1) > 0, ws[1].reshape(b, -1) > 0
    dn2_local = onp.bf16_round((ws[3].astype(np.float64).reshape(b, -1) @ f["w1"].T) * n2_mask)
    dn1_local = go.col2im(ws[4].astype(np.float64).reshape(-1, 32) @ f["w12"].T, b, g.h1, g.w1, 4, 2, g.h2, g.w2, 16)
    dn1_local = onp.bf16_round(dn1_local.reshape(b, -1) * n1_mask)
    rep["dn2"], rep["dn2_local"] = err(ws[4], f["dn2"]), err(ws[4], dn2_local)
    rep["dn1"], rep["dn1_local"] = err(ws[5], f["dn1"]), err(ws[5], dn1_local)
    for k, i in (("dn1", 5), ("dn2", 4)):
        ref = np.asarray(f[k], dtype=np.float64).ravel()
        rep[k + "_outliers"] = (float((np.abs(ws[i].ravel() - ref) > 2.0 ** -7 * np.abs(ref).max()).mean()), 0.0)
    for k in ("cost_p_1", "cost_p_2", "cost_v", "cost_all"):
        rep["loss/" + k] = err([losses[k]], [losses_ref[k]])
    grads = net.get_gradients()
    for k in grads_ref:
        rep["grad/" + k] = err(grads[k], grads_ref[k])
    return rep


def check_report(rep):
    assert rep["p"][0] <= TOL_P and rep["v"][0] <= TOL_V, rep
    for k in ("n1", "n2", "dd1"):
        assert rep[k][1] <= TOL_ACT_REL, (k, rep[k])
    for k in ("dn2", "dn1"):
        assert rep[k + "_local"][1] <= TOL_ACT_REL, (k, rep[k + "_local"])
        assert rep[k][1] <= TOL_ACT_REL or rep[k + "_outliers"][0] <= 1e-4, (k, rep[k], rep[k + "_outliers"])
    assert rep["d1"][1] <= 1e-3, rep["d1"]
    for k, (d, r) in rep.items():
        if k.startswith("loss/"):
            assert r <= TOL_LOSS_REL or d <= 1e-5, (k, d, r)
        if k.startswith("grad/"):
            assert r <= TOL_GRAD_REL, (k, d, r)


@pytest.mark.parametrize("hwc", GEOMETRIES, ids=IDS)
def test_predict_matches_oracle(ga3c, hwc):
    g = go.Geometry(*hwc)
    net = make_net(ga3c, hwc, 300)
    for b in (1, 37, 300):
        params, _, x, _, _ = case(g, b, seed=b)
        net.set_variables(params)
        p, v = net.predict_p_and_v(x)
        pr, vr = go.forward(g, params, x, quant="bf16")
        assert np.abs(p - pr).max() <= TOL_P and np.abs(v - vr).max() <= TOL_V, (b, np.abs(p - pr).max(), np.abs(v - vr).max())


@pytest.mark.parametrize("hwc", GEOMETRIES, ids=IDS)
def test_layers_and_gradients_match_oracle(ga3c, hwc):
    """The 4 loss sums, all 10 gradients and the layer-local n1 / n2 / d1 / dd1 / dn2 / dn1 (row-major workspace)."""
    g = go.Geometry(*hwc)
    params, _, x, y_r, a = case(g, 37)
    net = make_net(ga3c, hwc, 64)
    assert net._table["dense1/w:0"][1] == (g.flat, 256) and net._table["conv11/w:0"][1] == (8, 8, hwc[2], 16)
    check_report(layer_report(net, g, params, x, y_r, a))


@pytest.mark.parametrize("hwc", GEOMETRIES, ids=IDS)
def test_train_steps_uint8_and_reruns(ga3c, hwc):
    """Three RMSProp steps: weights and slots against the oracle; uint8 frames give bit-identical results to their normalised
    fp32 copy; a second network fed the same steps ends bit-identical (fixed-order reductions)."""
    g = go.Geometry(*hwc)
    params, k, x, y_r, a = case(g, 29, seed=5)
    lr = 3e-4
    results = []
    for frames in (x, k, x):
        net = make_net(ga3c, hwc, 32)
        net.set_variables(params)
        net.learning_rate = lr
        for _ in range(3):
            net.train(frames, y_r, a)
        results.append((net.get_variables(), net.get_slots()))
    p_ref = {kk: v.astype(np.float64) for kk, v in params.items()}
    ms, mom = onp.rmsprop_init(p_ref)
    for _ in range(3):
        _, grads = go.loss_and_grads(g, {kk: v.astype(np.float32) for kk, v in p_ref.items()}, x, y_r, a, quant="bf16")
        p_ref, ms, mom = onp.rmsprop_update(p_ref, grads, ms, mom, lr=lr, dtype=np.float64)
    w, (gms, gmom) = results[0]
    for kk in params:
        # each step's update carries at most TOL_W_ABS of error (test_gpu_parity.py), three steps three times that
        assert np.abs(w[kk] - p_ref[kk]).max() <= 3 * TOL_W_ABS, (kk, np.abs(w[kk] - p_ref[kk]).max())
        assert np.abs(gms[kk] - ms[kk]).max() <= 1e-3 * max(np.abs(ms[kk]).max(), 1e-30) + 1e-9, kk
    for other in results[1:]:
        for kk in params:
            assert np.array_equal(results[0][0][kk], other[0][kk]), kk
            assert np.array_equal(results[0][1][0][kk], other[1][0][kk]), kk


def test_predict_uint8_bit_identical(ga3c):
    hwc = (105, 80, 4)
    g = go.Geometry(*hwc)
    params, k, x, _, _ = case(g, 41)
    net = make_net(ga3c, hwc, 64)
    net.set_variables(params)
    p, v = net.predict_p_and_v(x)
    p8, v8 = net.predict_p_and_v(k)
    assert np.array_equal(p, p8) and np.array_equal(v, v8)


def test_b1024_training_matches_oracle(ga3c):
    hwc = (42, 42, 4)
    g = go.Geometry(*hwc)
    params, _, x, y_r, a = case(g, 1024, seed=1024)
    net = make_net(ga3c, hwc, 1024)
    check_report(layer_report(net, g, params, x, y_r, a))
    net.train(x, y_r, a)
    assert all(np.isfinite(v).all() for v in net.get_variables().values())


def test_log_softmax_min_policy(ga3c):
    hwc = (84, 84, 3)
    g = go.Geometry(*hwc)
    params, _, x, y_r, a = case(g, 33)
    net = make_net(ga3c, hwc, 64, USE_LOG_SOFTMAX=True)
    check_report(layer_report(net, g, params, x, y_r, a, use_log_softmax=True))
    net = make_net(ga3c, hwc, 64, MIN_POLICY=0.05)
    check_report(layer_report(net, g, params, x, y_r, a, min_policy=0.05))


def test_grad_clip_and_dual_rmsprop(ga3c):
    hwc = (100, 100, 2)
    g = go.Geometry(*hwc)
    params, _, x, y_r, a = case(g, 20)
    lr = 3e-4
    # USE_GRAD_CLIP: clip_by_average_norm per variable before RMSProp
    net = make_net(ga3c, hwc, 32, USE_GRAD_CLIP=True, GRAD_CLIP_NORM=0.05)
    net.set_variables(params)
    net.learning_rate = lr
    net.train(x, y_r, a)
    _, grads = go.loss_and_grads(g, params, x, y_r, a, quant="bf16")
    ref = {k: v.astype(np.float64) for k, v in params.items()}
    ms, mom = onp.rmsprop_init(ref)
    p2, _, _ = onp.rmsprop_update(ref, {k: onp.clip_by_average_norm(v, 0.05) for k, v in grads.items()}, ms, mom, lr=lr,
                                  dtype=np.float64)
    w = net.get_variables()
    for k in params:
        assert np.abs(w[k] - p2[k]).max() <= TOL_W_ABS, k
    # DUAL_RMSPROP: both steps from the pre-call weights
    net = make_net(ga3c, hwc, 32, DUAL_RMSPROP=True)
    net.set_variables(params)
    net.learning_rate = lr
    net.train(x, y_r, a)
    new = {k: v.astype(np.float64) for k, v in params.items()}
    for part in ("p", "v"):
        _, gp = go.loss_and_grads(g, params, x, y_r, a, quant="bf16", part=part)
        sub = {k: params[k].astype(np.float64) for k in gp}
        ms, mom = onp.rmsprop_init(sub)
        p2, _, _ = onp.rmsprop_update(sub, gp, ms, mom, lr=lr, dtype=np.float64)
        for k in gp:
            new[k] -= params[k] - p2[k]
    w = net.get_variables()
    for k in params:
        assert np.abs(w[k] - new[k]).max() <= TOL_W_ABS, k


def test_histograms_match_oracle(ga3c):
    hwc = (105, 80, 4)
    g = go.Geometry(*hwc)
    params, _, x, y_r, a = case(g, 24)
    net = make_net(ga3c, hwc, 32)
    net.set_variables(params)
    stats = net.histograms(x, y_r, a)
    b = x.shape[0]
    n1, n2, d1 = net.workspace(0), net.workspace(1), net.workspace(2)
    p, v = net.predict_p_and_v(x)
    want = dict(zip(net._hist_tags[-5:], (n1, n2, d1, v, p)))
    want.update({t: params[k] for t, k in zip(net._hist_tags[:10], net._table)})
    for tag, vals in want.items():
        ref = hnp.histogram(np.asarray(vals, dtype=np.float64).ravel())
        got = stats[tag]
        assert got[2] == ref[2] and np.array_equal(np.asarray(got[5]), np.asarray(ref[5])), tag
        assert got[0] == ref[0] and got[1] == ref[1], tag
    assert n1.size == b * g.h1 * g.w1 * 16 and n2.size == b * g.flat


def test_save_load_roundtrip_and_cross_geometry_load(ga3c, tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    hwc = (8, 8, 1)
    g = go.Geometry(*hwc)
    params, _, x, y_r, a = case(g, 9)
    net = make_net(ga3c, hwc, 16)
    net.set_variables(params)
    net.train(x, y_r, a)
    net.save(3)
    other = make_net(ga3c, hwc, 16)
    assert other.load() == 3
    for k, v in net.get_variables().items():
        assert np.array_equal(other.get_variables()[k], v)
    for mine, theirs in zip(net.get_slots(), other.get_slots()):
        for k in mine:
            assert np.array_equal(mine[k], theirs[k])
    wrong = make_net(ga3c, (16, 8, 1), 16)
    with pytest.raises(ValueError, match="dense1/w"):
        wrong.load()


def test_default_geometry_runs_only_the_specialised_kernels(ga3c):
    params, x, y_r, a = onp.init_params(np.random.default_rng(0), 6), onp.synth_frames(np.random.default_rng(1), 16), \
        *onp.synth_targets(np.random.default_rng(2), 16, 6)
    net = ga3c.Network("gpu:0", "geo", 6, max_batch=16)
    net.set_variables(params)
    net.kernel_timing(256)
    net.predict_p_and_v(x)
    net.train(x, y_r, a)
    names = set(net.kernel_times())
    assert "conv_fwd" in names and "conv_bwd" in names and not names & GEN_KERNELS, names
    gen = make_net(ga3c, (84, 84, 2), 16)
    gen.kernel_timing(256)
    gen.train(onp.synth_frames(np.random.default_rng(1), 16)[:, : 84 * 84 * 2], y_r, a)
    names = set(gen.kernel_times())
    assert GEN_KERNELS <= names and "conv_fwd" not in names and "conv_bwd" not in names, names


@pytest.mark.parametrize("knob,value", [("IMAGE_HEIGHT", 0), ("IMAGE_HEIGHT", 257), ("IMAGE_WIDTH", 0), ("IMAGE_WIDTH", 300),
                                        ("STACKED_FRAMES", 9), ("STACKED_FRAMES", 0)])
def test_out_of_range_knobs_are_refused(ga3c, knob, value):
    """Network refuses the knob by name, with state_dim left to its default (H*W*C) too; ga3c_create refuses a non-zero value out
    of range by its field name (0 there means the default 84 / 84 / 4)."""
    import ctypes as C
    from ga3c_b200 import _capi
    hwc = {"IMAGE_HEIGHT": 84, "IMAGE_WIDTH": 84, "STACKED_FRAMES": 4}
    hwc[knob] = value
    cfg = config((hwc["IMAGE_HEIGHT"], hwc["IMAGE_WIDTH"], hwc["STACKED_FRAMES"]))
    with pytest.raises(ValueError, match=knob):
        ga3c.Network("gpu:0", "geo", 6, config=cfg, max_batch=8)
    with pytest.raises(ValueError, match=knob):
        ga3c.Network("gpu:0", "geo", 6, max(1, hwc["IMAGE_HEIGHT"] * hwc["IMAGE_WIDTH"] * hwc["STACKED_FRAMES"]), config=cfg,
                     max_batch=8)
    if value:
        field = {"IMAGE_HEIGHT": "image_height", "IMAGE_WIDTH": "image_width", "STACKED_FRAMES": "stacked_frames"}[knob]
        c = _capi.ga3c_config(device=0, num_actions=6, max_batch=8, rmsprop_decay=0.99, rmsprop_epsilon=0.1, log_epsilon=1e-6,
                              grad_clip_norm=40.0, **{field: value})
        h = C.c_void_p()
        lib = _capi.load()
        assert lib.ga3c_create(C.byref(c), C.byref(h)) != 0 and not h.value
        msg = lib.ga3c_last_error().decode()
        assert field in msg and knob in msg, msg


def test_state_dim_mismatch_raises(ga3c):
    with pytest.raises(ValueError, match="STACKED_FRAMES"):
        ga3c.Network("gpu:0", "geo", 6, 84 * 84 * 4, config=config((84, 84, 2)), max_batch=8)


def test_predictors_and_trainer_over_the_slab_transport(ga3c):
    """ThreadPredictor, NativePredictor and ThreadTrainer serve a 42x42x4 uint8 network through the slab queues; the native
    batcher refuses a frame row that is not a multiple of 16 bytes."""
    import time
    from ga3c_b200.transport import SlabPredictionQueue, SlabTrainingQueue
    from test_gpu_parity import _Server
    hwc, n = (42, 42, 4), 24
    g = go.Geometry(*hwc)
    params, k, x, y_r, a = case(g, n)
    net = make_net(ga3c, hwc, 64)
    net.set_variables(params)
    pr, vr = go.forward(g, params, x, quant="bf16")
    for native in (False, True):
        net.set_variables(params)             # the trainer of the previous round moved them
        pq = SlabPredictionQueue(n, g.state_dim, 6, dtype=np.uint8)
        tq = SlabTrainingQueue(n, max_rows=4, state_dim=g.state_dim, num_actions=6, dtype=np.uint8)
        srv = _Server(net, n)
        srv.training_q = tq
        pred = ga3c.NativePredictor(srv, 0, pq) if native else ga3c.ThreadPredictor(srv, 0, g.state_dim, pq)

        class Cfg(ga3c.Config):
            TRAINING_MIN_BATCH_SIZE = 10
        tr = ga3c.ThreadTrainer(srv, 0, config=Cfg)
        pred.start(); tr.start()
        try:
            pq.post_many(np.arange(n), k)
            p = np.zeros((n, 6), np.float32); v = np.zeros(n, np.float32)
            assert pq.wait_many(np.arange(n), p, v, timeout=60) == n
            assert np.abs(p - pr).max() <= TOL_P and np.abs(v - vr).max() <= TOL_V
            for i in range(0, 12, 4):
                tq.for_agent(i).put((k[i:i + 4], y_r[i:i + 4].astype(np.float64), a[i:i + 4], k[i:i + 4], np.zeros(4, bool)))
            t0 = time.time()
            while not srv.trained and time.time() - t0 < 60:
                time.sleep(0.01)
            assert srv.trained and srv.trained[0] == 12
        finally:
            pred.exit_flag = True; tr.exit_flag = True
            time.sleep(0.2)
            if native:
                pred.close()
            pq.close(); tq.close()
    small = make_net(ga3c, (5, 5, 1), 8)
    pq = SlabPredictionQueue(2, 25, 6, dtype=np.uint8)
    try:
        with pytest.raises(ga3c._capi.Ga3cError, match="multiple of 16 bytes"):
            ga3c.NativePredictor(_Server(small, 2), 0, pq)
    finally:
        pq.close()


def _dev(*arrays):
    import torch
    return [torch.as_tensor(np.ascontiguousarray(v)).cuda() for v in arrays]


@pytest.mark.parametrize("u8", [False, True], ids=["fp32", "uint8"])
def test_fb_head_and_fb_tail_match_oracle(ga3c, u8):
    """The split entry points a data-parallel host (dp_mode 'nccl') calls: ga3c_fb_head (forward, heads and dense1's weight
    gradient at the handle's K) then ga3c_fb_tail (dense1's data gradient alone, row-major dn2, and the conv backward).  All 10
    gradients and the loss sums against the bf16 oracle, and equal bit for bit to ga3c_forward_backward."""
    import torch
    from ga3c_b200 import _capi
    hwc = (105, 80, 4)
    g = go.Geometry(*hwc)
    params, k, x, y_r, a = case(g, 45, seed=9)
    net = make_net(ga3c, hwc, 64)
    net.set_variables(params)
    dx, dyr, da = _dev(k if u8 else x, y_r, a)
    loss = torch.zeros(4, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    head = net._lib.ga3c_fb_head_u8 if u8 else net._lib.ga3c_fb_head
    tail = net._lib.ga3c_fb_tail_u8 if u8 else net._lib.ga3c_fb_tail
    _capi.check(head(net._h, dx.data_ptr(), dyr.data_ptr(), da.data_ptr(), 45, float(net.beta), loss.data_ptr(), st), "fb_head")
    _capi.check(tail(net._h, dx.data_ptr(), 45, st), "fb_tail")
    torch.cuda.synchronize()
    split = net.get_gradients()
    losses = net._loss_dict(loss.cpu())
    losses_ref, grads_ref = go.loss_and_grads(g, params, x, y_r, a, quant="bf16", beta=net.beta)
    for kk in ("cost_p_1", "cost_p_2", "cost_v", "cost_all"):
        d, r = err([losses[kk]], [losses_ref[kk]])
        assert r <= TOL_LOSS_REL or d <= 1e-5, (kk, d, r)
    for kk in grads_ref:
        assert err(split[kk], grads_ref[kk])[1] <= TOL_GRAD_REL, (kk, err(split[kk], grads_ref[kk]))
    net.losses(k if u8 else x, y_r, a)                  # ga3c_forward_backward on the same rows
    whole = net.get_gradients()
    for kk in whole:
        assert np.array_equal(whole[kk], split[kk]), kk


def test_reserve_failure_leaves_a_usable_handle(ga3c):
    """ga3c_reserve at a batch whose generic workspace cannot be allocated (256x256x8: 4.3 MB of im2col per row) returns an error;
    the handle then refuses every batch, and a later reserve that fits brings it back."""
    import ctypes as C
    hwc = (256, 256, 8)
    g = go.Geometry(*hwc)
    params, _, x, _, _ = case(g, 3)
    net = make_net(ga3c, hwc, 4)
    net.set_variables(params)
    assert net._lib.ga3c_reserve(net._h, 2_000_000) != 0
    assert "cudaMalloc" in net._lib.ga3c_last_error().decode()
    import torch
    p, v = torch.empty((3, 6), device="cuda"), torch.empty(3, device="cuda")
    xd, = _dev(x)
    assert net._lib.ga3c_predict(net._h, xd.data_ptr(), 3, p.data_ptr(), v.data_ptr(), None) != 0
    assert "batch 3 outside" in net._lib.ga3c_last_error().decode()
    assert net._lib.ga3c_reserve(net._h, 8) == 0
    assert net._lib.ga3c_predict(net._h, xd.data_ptr(), 3, p.data_ptr(), v.data_ptr(), None) == 0
    torch.cuda.synchronize()
    pr, vr = go.forward(g, params, x, quant="bf16")
    assert np.abs(p.cpu().numpy() - pr).max() <= TOL_P and np.abs(v.cpu().numpy() - vr).max() <= TOL_V


def test_nccl_data_parallel_step_two_gpus(ga3c):
    """Two ranks, one GPU each, at 42x42x4: Network switches to dp_mode 'nccl'; after three steps on row shards the replicas are
    bit-identical and match the oracle's steps on the whole batch.  Needs >= 2 visible GPUs."""
    import os
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    here = os.path.dirname(os.path.abspath(__file__))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
                        "127.0.0.1", "--master-port", "29613", os.path.join(here, "dp_geometry_torchrun.py")],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "DP_GEOMETRY OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
