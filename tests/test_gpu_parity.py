"""GPU parity tests (`-m gpu`): the CUDA path, called through the C-ABI library, against the oracle.

Tolerances: tests/_parity.py.  Integer / fp64 work (returns, sampling) is bit-exact.
"""
import json
import os
import threading
import queue

import numpy as np
import pytest

from oracle import oracle_np as onp
from _parity import TOL_GRAD_REL, TOL_LOSS_REL, TOL_P, TOL_V, TOL_W_ABS, check_report, err, layer_report, make_case
from _parity import ga3c  # noqa: F401  (pytest fixture)

pytestmark = pytest.mark.gpu


# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("batch", [1, 2, 7, 32, 33, 128, 300])
def test_layers_and_gradients_match_oracle(ga3c, batch):
    """Every stored activation, all 10 gradients and the 4 loss sums, at ragged and full batch sizes
    (1, odd, one CTA chunk +1, PREDICTION_BATCH_SIZE, more than 2 x 148 CTAs)."""
    params, x, y_r, a = make_case(batch)
    net = ga3c.Network("gpu:0", "t", 6, max_batch=max(batch, 16))
    check_report(layer_report(net, params, x, y_r, a))


def test_layers_and_gradients_match_oracle_b1024(ga3c):
    """The benchmarked train shape (BASELINE configs[2], B = 1024 per GPU: 7 rounds of frames per persistent conv CTA, split-K
    factor of that batch): every stored activation, all 10 gradients and the loss sums of the FULL batch against the oracle."""
    params, x, y_r, a = make_case(1024, seed=1024)
    net = ga3c.Network("gpu:0", "t", 6, max_batch=1024)
    check_report(layer_report(net, params, x, y_r, a))


def test_predict_b4096_full_batch_matches_oracle(ga3c):
    """The benchmarked predict shape (configs[1], B = 4096): every row of p and v against the oracle."""
    rng = np.random.default_rng(40960)
    params = onp.init_params(rng, 6)
    x = onp.synth_frames(rng, 4096)
    net = ga3c.Network("gpu:0", "t", 6, max_batch=4096)
    net.set_variables(params)
    p, v = net.predict_p_and_v(x)
    pr, vr = onp.forward(params, x, quant="bf16")
    assert np.abs(p - pr).max() <= TOL_P and np.abs(v - vr).max() <= TOL_V, (np.abs(p - pr).max(), np.abs(v - vr).max())


@pytest.mark.parametrize("batch", [8, 32, 160])
def test_back_to_back_async_steps_equal_synchronised_steps(ga3c, batch):
    """The asynchronous API (train_device / the C-ABI on one stream, no host synchronisation between calls): N steps enqueued
    back to back leave bit-identical weights and slots to the same steps with a device synchronisation after each.  With a
    batch below the SM count every kernel of a step fits next to the previous step's optimizer launch, which is where a
    prologue that read mutable state before its dependency wait would see a half-applied update."""
    import torch
    rng = np.random.default_rng(batch)
    params = onp.init_params(rng, 6)
    steps = 12
    data = [(onp.synth_frames(rng, batch),) + onp.synth_targets(rng, batch) for _ in range(3)]
    results = []
    for sync in (True, False):
        net = ga3c.Network("gpu:0", "t", 6, max_batch=max(batch, 16))
        net.set_variables(params)
        dev = [[torch.as_tensor(t).cuda() for t in d] for d in data]
        p_out = [torch.empty((batch, 6), device="cuda") for _ in range(steps)]
        v_out = [torch.empty((batch,), device="cuda") for _ in range(steps)]
        torch.cuda.synchronize()
        st = torch.cuda.current_stream()
        for i in range(steps):
            net.train_device(*dev[i % 3], stream=st)
            net.predict_device(dev[(i + 1) % 3][0], p_out[i], v_out[i], stream=st)      # predict-after-train on the same stream
            if sync:
                torch.cuda.synchronize()
        torch.cuda.synchronize()
        results.append((net.get_variables(), net.get_slots()[0], [t.cpu().numpy() for t in p_out], [t.cpu().numpy() for t in v_out]))
    (w0, m0, p0, v0), (w1, m1, p1, v1) = results
    for k in w0:
        assert np.array_equal(w0[k], w1[k]) and np.array_equal(m0[k], m1[k]), k
    assert all(np.array_equal(a_, b_) for a_, b_ in zip(p0, p1)) and all(np.array_equal(a_, b_) for a_, b_ in zip(v0, v1))


@pytest.mark.parametrize("num_actions", [1, 2, 18])
def test_num_actions_range(ga3c, num_actions):
    params, x, y_r, a = make_case(9, num_actions=num_actions, seed=3)
    net = ga3c.Network("gpu:0", "t", num_actions, max_batch=16)
    check_report(layer_report(net, params, x, y_r, a))


def test_min_policy_and_active_epsilon_floor(ga3c):
    """MIN_POLICY mixing and an epsilon floor large enough that both mask branches of A.4 fire."""
    class Cfg(ga3c.Config):
        MIN_POLICY = 0.02
        LOG_EPSILON = 0.16
    params, x, y_r, a = make_case(24, seed=11)
    params["logits_p/w:0"] *= 8.0           # spread the policy so some p_ij fall under the floor
    net = ga3c.Network("gpu:0", "t", 6, max_batch=32, config=Cfg)
    rep = layer_report(net, params, x, y_r, a, beta=0.05, log_eps=0.16, min_policy=0.02)
    p, _ = onp.forward(params, x, quant="bf16", min_policy=0.02)
    assert (p < 0.16).any() and (p >= 0.16).any()
    check_report(rep)


def test_log_softmax_knob(ga3c):
    """Config.USE_LOG_SOFTMAX = True (NetworkVP_discrate.py:64-71): log_softmax losses, plain softmax policy (MIN_POLICY and
    the epsilon floor do not apply); every activation, gradient and loss sum against the oracle's same branch."""
    class Cfg(ga3c.Config):
        USE_LOG_SOFTMAX = True
        MIN_POLICY = 0.02
    params, x, y_r, a = make_case(40, seed=13)
    params["logits_p/w:0"] *= 6.0
    net = ga3c.Network("gpu:0", "t", 6, max_batch=64, config=Cfg)
    rep = layer_report(net, params, x, y_r, a, beta=0.05, use_log_softmax=True)
    check_report(rep)
    p, _ = net.predict_p_and_v(x)
    assert np.allclose(p.sum(axis=1), 1.0, atol=1e-5)


def test_data_parallel_exchange_two_ranks_on_one_gpu(ga3c, monkeypatch):
    """The fused data-parallel step (dp_exchange.cuh: dense1/w exchanged by a small-footprint kernel on a side stream next to
    the conv kernels, LL push of the small tensors after the conv backward) with BOTH ranks on one device: two handles attached
    to each other with ga3c_dp_attach_local, each on its own stream, each training on its row shard.  After 3 steps the replicas
    are bit-identical and equal the oracle's single-process steps on the concatenated batch (what a single ThreadTrainer would
    have computed).  The grids are small (12 rows per rank), so both ranks' kernels are resident together; every cross-rank
    wait is bounded, so a scheduling surprise fails the test instead of hanging the GPU.  ga3c_apply_rmsprop refuses an
    attached handle: its exchange is part of ga3c_train_step."""
    import ctypes as C
    import torch
    from ga3c_b200 import _capi
    monkeypatch.setenv("GA3C_DP_SIDE_CTAS", "8")      # both ranks share this GPU: leave room for the other rank's conv kernels
    world, b = 2, 12
    rng = np.random.default_rng(17)
    params = onp.init_params(rng, 6)
    nets = [ga3c.Network("gpu:0", f"dp{r}", 6, max_batch=32, data_parallel=False) for r in range(world)]
    lib = _capi.load()
    handles = (C.c_void_p * world)(*[n._h.value for n in nets])
    try:
        for n in nets:
            n.set_variables(params)
        for r, n in enumerate(nets):
            _capi.check(lib.ga3c_dp_attach_local(n._h, r, world, handles), "ga3c_dp_attach_local")
        streams = [torch.cuda.Stream() for _ in nets]
        ms, mom = onp.rmsprop_init(params)
        ref = params
        for step in range(3):
            x = onp.synth_frames(rng, world * b)
            y_r, a = onp.synth_targets(rng, world * b)
            dev = [[torch.as_tensor(t[r * b:(r + 1) * b]).cuda() for t in (x, y_r, a)] for r in range(world)]
            torch.cuda.synchronize()
            for r, n in enumerate(nets):         # asynchronous: both ranks' kernels must be in flight together
                n.train_device(*dev[r], stream=streams[r])
            torch.cuda.synchronize()
            _, _, ref, ms, mom = onp.train_step(ref, ms, mom, x, y_r, a, lr=nets[0].learning_rate, beta=nets[0].beta, quant="bf16")
            ref = {k: v.astype(np.float32) for k, v in ref.items()}
        # a lock-step round in which rank 1 has nothing to train on: it enters the step with batch = 0 (zero gradient) and
        # applies the same update -- equal to the oracle's step on rank 0's rows alone
        x = onp.synth_frames(rng, b)
        y_r, a = onp.synth_targets(rng, b)
        d0 = [torch.as_tensor(t).cuda() for t in (x, y_r, a)]
        d1 = [torch.as_tensor(t[:0]).cuda() for t in (x, y_r, a)]
        torch.cuda.synchronize()
        nets[0].train_device(*d0, stream=streams[0])
        nets[1].train_device(*d1, stream=streams[1])
        torch.cuda.synchronize()
        _, _, ref, ms, mom = onp.train_step(ref, ms, mom, x, y_r, a, lr=nets[0].learning_rate, beta=nets[0].beta, quant="bf16")
        ref = {k: v.astype(np.float32) for k, v in ref.items()}
        for n in nets:
            n.dp_check()
        w = [n.get_variables() for n in nets]
        m = [n.get_slots()[0] for n in nets]
        sh = [n.workspace(6) for n in nets]
        assert np.array_equal(sh[0], sh[1])                                                     # the bf16 shadow every rank holds
        for k in params:
            assert np.array_equal(w[0][k], w[1][k]) and np.array_equal(m[0][k], m[1][k]), k     # replicas bit-identical
            assert np.abs(w[0][k] - ref[k]).max() <= 4 * TOL_W_ABS, (k, np.abs(w[0][k] - ref[k]).max())
        assert nets[0].get_global_step() == 4 and nets[1].get_global_step() == 4
        assert lib.ga3c_apply_rmsprop(nets[0]._h, C.c_float(1e-3), None) != 0
        assert b"ga3c_train_step" in lib.ga3c_last_error()
    finally:
        for n in nets:
            lib.ga3c_dp_detach(n._h)


def test_grad_clip_knob(ga3c):
    """Config.USE_GRAD_CLIP = True (NetworkVP_discrate.py:118-121): tf.clip_by_average_norm per variable before RMSProp, with a
    threshold small enough to be active on some variables and not on others; as in the reference file the step counter is
    not advanced (apply_gradients is called without global_step)."""
    clip = 2e-5
    class Cfg(ga3c.Config):
        USE_GRAD_CLIP = True
        GRAD_CLIP_NORM = clip
    params, x, y_r, a = make_case(48, seed=19)
    net = ga3c.Network("gpu:0", "t", 6, max_batch=64, config=Cfg)
    net.set_variables(params)
    ms, mom = onp.rmsprop_init(params)
    ref = params
    for step in range(2):
        net.train(x, y_r, a, None, None, 0)
        _, grads, ref, ms, mom = onp.train_step(ref, ms, mom, x, y_r, a, lr=net.learning_rate, beta=net.beta, quant="bf16",
                                                grad_clip=clip)
        ref = {k: v.astype(np.float32) for k, v in ref.items()}
    avg = {k: np.sqrt((g.astype(np.float64) ** 2).sum()) / g.size for k, g in grads.items()}
    assert any(v > clip for v in avg.values()) and any(v < clip for v in avg.values()), avg
    got = net.get_variables()
    for k in got:
        assert np.abs(got[k] - ref[k]).max() <= TOL_W_ABS, (k, np.abs(got[k] - ref[k]).max())
    assert net.get_global_step() == 0


def test_dual_rmsprop_knob(ga3c):
    """Config.DUAL_RMSPROP = True (NetworkVP_discrate.py:87-98, :124-128): cost_p and cost_v minimised by two RMSProp optimizers.
    Both gradients at the pre-call weights, both steps subtracted (the order-independent reading of TF's two train ops);
    each optimizer's own ms slots; logits_v untouched by the cost_p optimizer and logits_p by the cost_v one; global_step += 2."""
    class Cfg(ga3c.Config):
        DUAL_RMSPROP = True
    params, x, y_r, a = make_case(40, seed=23)
    net = ga3c.Network("gpu:0", "t", 6, max_batch=64, config=Cfg)
    net.set_variables(params)
    ms, mom = onp.rmsprop_init(params)
    ref, sp, sv = params, (ms, mom), (ms, mom)
    for step in range(3):
        got = net.train(x, y_r, a, None, None, 0, fetch_losses=True)
        losses, gp, gv, ref, sp, sv = onp.train_step_dual(ref, sp, sv, x, y_r, a, lr=net.learning_rate, beta=net.beta, quant="bf16")
        ref = {k: v.astype(np.float32) for k, v in ref.items()}
        assert abs(got["cost_all"] - losses["cost_all"]) <= TOL_LOSS_REL * max(1.0, abs(losses["cost_all"]))
    w = net.get_variables()
    for k in w:
        assert np.abs(w[k] - ref[k]).max() <= 2 * TOL_W_ABS, (k, np.abs(w[k] - ref[k]).max())
    ms_p, _ = net.get_slots(0)
    ms_v, _ = net.get_slots(1)
    for k in w:
        assert err(ms_p[k], sp[0][k])[1] <= 2e-3 and err(ms_v[k], sv[0][k])[1] <= 2e-3, k
    assert np.array_equal(ms_p["logits_v/w:0"], np.ones_like(ms_p["logits_v/w:0"]))      # never touched by the cost_p optimizer
    assert np.array_equal(ms_v["logits_p/w:0"], np.ones_like(ms_v["logits_p/w:0"]))
    assert net.get_global_step() == 6
    g_p, g_v = net._split(net._download(1)), net._split(net._download(4))
    for k in gp:
        assert err(g_p[k], gp[k])[1] <= TOL_GRAD_REL, (k, err(g_p[k], gp[k]))
    for k in gv:
        assert err(g_v[k], gv[k])[1] <= TOL_GRAD_REL, (k, err(g_v[k], gv[k]))


def test_dual_rmsprop_with_grad_clip(ga3c):
    """Config.DUAL_RMSPROP + USE_GRAD_CLIP (NetworkVP_discrate.py:107-117): tf.clip_by_norm per variable on each optimizer's
    gradients (threshold chosen so that it is active on some variables and not on others), two RMSProp steps from the
    pre-call weights, and no global_step (apply_gradients is called without it)."""
    clip = 2.0
    class Cfg(ga3c.Config):
        DUAL_RMSPROP = True
        USE_GRAD_CLIP = True
        GRAD_CLIP_NORM = clip
    params, x, y_r, a = make_case(40, seed=31)
    net = ga3c.Network("gpu:0", "t", 6, max_batch=64, config=Cfg)
    net.set_variables(params)
    ms, mom = onp.rmsprop_init(params)
    ref, sp, sv = params, (ms, mom), (ms, mom)
    for step in range(2):
        net.train(x, y_r, a, None, None, 0)
        _, gp, gv, ref, sp, sv = onp.train_step_dual(ref, sp, sv, x, y_r, a, lr=net.learning_rate, beta=net.beta, quant="bf16",
                                                     grad_clip=clip)
        ref = {k: v.astype(np.float32) for k, v in ref.items()}
    norms = [float(np.sqrt((g.astype(np.float64) ** 2).sum())) for g in list(gp.values()) + list(gv.values())]
    assert any(v > clip for v in norms) and any(v < clip for v in norms), norms
    w = net.get_variables()
    for k in w:
        assert np.abs(w[k] - ref[k]).max() <= 2 * TOL_W_ABS, (k, np.abs(w[k] - ref[k]).max())
    ms_p, _ = net.get_slots(0)
    ms_v, _ = net.get_slots(1)
    for k in w:                                # ms = 0.99^2 + O(g_clipped^2): compared absolutely (fp32 slots)
        assert np.abs(ms_p[k] - sp[0][k]).max() <= 1e-6 and np.abs(ms_v[k] - sv[0][k]).max() <= 1e-6, k
    assert np.array_equal(ms_p["logits_v/w:0"], np.ones_like(ms_p["logits_v/w:0"]))      # never touched by the cost_p optimizer
    assert net.get_global_step() == 0


def test_log_writes_the_reference_scalars(ga3c, tmp_path, monkeypatch):
    """Network.log (NetworkVP.py:259-265; called by Server.py:149-150 every TENSORBOARD_UPDATE_FREQUENCY steps): a second
    forward pass that records Pcost_advantage, Pcost_entropy, Pcost, Vcost, LearningRate, Beta -- and leaves the weights,
    the slots and the step counter alone."""
    monkeypatch.chdir(tmp_path)
    params, x, y_r, a = make_case(24, seed=41)
    net = ga3c.Network("gpu:0", "logtest", 6, max_batch=32)
    net.set_variables(params)
    net.learning_rate, net.beta = 1e-4, 0.02
    net.log(x, y_r, a, 7)
    net.log(x[:5], y_r[:5], a[:5], 8)
    rows = [l.strip().split(",") for l in open(tmp_path / "logs" / "logtest" / "scalars.csv")]
    assert [int(r[0]) for r in rows] == [7, 8] and all(len(r) == 7 for r in rows)
    l_ref, _ = onp.loss_and_grads(params, x, y_r, a, beta=0.02, quant="bf16")
    got = [float(v) for v in rows[0][1:]]
    want = [l_ref["cost_p_1"], l_ref["cost_p_2"], l_ref["cost_p"], l_ref["cost_v"], 1e-4, 0.02]
    assert np.allclose(got, want, rtol=TOL_LOSS_REL, atol=1e-5), (got, want)
    w = net.get_variables()
    assert all(np.array_equal(w[k], params[k]) for k in w) and net.get_global_step() == 0


def test_slab_transport_feeds_the_cuda_network(ga3c):
    """8f F1 on the GPU: agents post uint8 frames into the shared-memory slab queue, ga3c_b200.ThreadPredictor gathers them
    into its pinned batch and calls the CUDA Network, replies travel back through the slab; the trainer path likewise.  Every
    reply equals the oracle's prediction for the frame that agent posted."""
    import time
    from ga3c_b200.transport import SlabPredictionQueue, SlabTrainingQueue
    n_agents = 48
    rng = np.random.default_rng(51)
    params = onp.init_params(rng, 6)
    k = rng.integers(0, 256, size=(n_agents, onp.STATE_DIM), dtype=np.uint8)
    x = k.astype(np.float32) / 128.0 - 1.0
    y_r, a = onp.synth_targets(rng, n_agents)
    net = ga3c.Network("gpu:0", "t", 6, max_batch=128)
    net.set_variables(params)
    pq = SlabPredictionQueue(n_agents, onp.STATE_DIM, 6, dtype=np.uint8)
    tq = SlabTrainingQueue(n_agents, max_rows=4, state_dim=onp.STATE_DIM, num_actions=6, dtype=np.uint8)
    srv = _Server(net, n_agents)
    srv.training_q = tq
    pred = ga3c.ThreadPredictor(srv, 0, onp.STATE_DIM, pq)
    class Cfg(ga3c.Config):
        TRAINING_MIN_BATCH_SIZE = 30
    tr = ga3c.ThreadTrainer(srv, 0, config=Cfg)
    pred.start(); tr.start()
    try:
        pq.post_many(np.arange(n_agents), k)
        p = np.zeros((n_agents, 6), np.float32); v = np.zeros(n_agents, np.float32)
        assert pq.wait_many(np.arange(n_agents), p, v, timeout=60) == n_agents
        pr, vr = onp.forward(params, x, quant="bf16")
        assert np.abs(p - pr).max() <= TOL_P and np.abs(v - vr).max() <= TOL_V
        assert pred.rows == n_agents
        for i in range(0, n_agents, 4):                                     # 12 agent batches of 4 rows
            tq.for_agent(i).put((k[i:i + 4], y_r[i:i + 4].astype(np.float64), a[i:i + 4], k[i:i + 4], np.zeros(4, bool)))
        t0 = time.time()
        while sum(srv.trained) < 32 and time.time() - t0 < 60:
            time.sleep(0.01)
        assert srv.trained and srv.trained[0] == 32                         # 8 x 4 rows: the first count that EXCEEDS 30
        assert net.get_global_step() >= 1
    finally:
        pred.exit_flag = True; tr.exit_flag = True
        time.sleep(0.2)
        pq.close(); tq.close()


@pytest.mark.parametrize("dtype", [np.uint8, np.float32])
def test_native_predictor_batcher_over_the_slab(ga3c, dtype):
    """The predictor loop inside the library (ga3c_batcher_*, ga3c_b200.NativePredictor): requests posted into the slab are
    gathered from the page-locked state rows by a kernel, predicted, and answered on the agents' own wait_q -- every reply equals
    the oracle's prediction for the frame that agent posted, over several rounds, while a trainer thread trains on the same
    network (the handle's mutex serialises them)."""
    import time
    from ga3c_b200.transport import SlabPredictionQueue
    n_agents, rounds = 200, 4
    rng = np.random.default_rng(61)
    params = onp.init_params(rng, 6)
    net = ga3c.Network("gpu:0", "t", 6, max_batch=128)
    net.set_variables(params)
    net.learning_rate = 0.0                              # weights stay put, so every round is checkable
    pq = SlabPredictionQueue(n_agents, onp.STATE_DIM, 6, dtype=dtype)
    srv = _Server(net, n_agents)
    pred = ga3c.NativePredictor(srv, 0, pq)
    pred.start()
    stop = threading.Event()
    xt = onp.synth_frames(rng, 32)
    yt, at = onp.synth_targets(rng, 32)

    def trainer():
        while not stop.is_set():
            net.train(xt, yt, at, None, None, 0)
    th = threading.Thread(target=trainer)
    th.start()
    try:
        for r in range(rounds):
            k = rng.integers(0, 256, size=(n_agents, onp.STATE_DIM), dtype=np.uint8)
            x = k.astype(np.float32) / 128.0 - 1.0
            pq.post_many(np.arange(n_agents), k if dtype == np.uint8 else x)
            p = np.zeros((n_agents, 6), np.float32); v = np.zeros(n_agents, np.float32)
            assert pq.wait_many(np.arange(n_agents), p, v, timeout=60) == n_agents
            pr, vr = onp.forward(params, x, quant="bf16")
            assert np.abs(p - pr).max() <= TOL_P and np.abs(v - vr).max() <= TOL_V, (r, np.abs(p - pr).max())
        assert pred.rows == n_agents * rounds and pred.batches >= 2 * rounds      # 200 pending rows: at least two batches of <= 128
        assert not pq._pending.array.any()
    finally:
        stop.set(); th.join()
        pred.exit_flag = True
        pred.close()
        pq.close()


def test_golden_network_b4(ga3c, golden_dir):
    """The committed B=4 fixture (tests/golden/network_b4.npz, oracle/gen_golden.py)."""
    g = np.load(os.path.join(golden_dir, "network_b4.npz"))
    params, x, y_r, a = make_case(4)
    net = ga3c.Network("gpu:0", "t", 6, max_batch=16)
    net.set_variables(params)
    p, v = net.predict_p_and_v(x)
    assert np.abs(p - g["bf16_p"]).max() <= TOL_P and np.abs(v - g["bf16_v"]).max() <= TOL_V
    assert np.abs(p - g["f64_p"]).max() <= 1e-2 and np.abs(v - g["f64_v"]).max() <= 2e-2     # bf16 gap
    l = net.losses(x, y_r, a)
    got = np.array([l[k] for k in ("cost_p_1", "cost_p_2", "cost_p", "cost_v", "cost_all")])
    assert np.allclose(got, g["bf16_losses"], rtol=TOL_LOSS_REL, atol=1e-5)
    grads = net.get_gradients()
    for k in ("conv11/b:0", "conv12/b:0", "dense1/b:0", "logits_p/w:0", "logits_v/w:0", "conv11/w:0"):
        ref = g["bf16_grad_" + k]
        assert err(grads[k], ref)[1] <= TOL_GRAD_REL, k


def test_prediction_is_fp32_softmax_accepted_by_numpy_choice(ga3c):
    """SURVEY A.6: np.random.choice rejects p whose sum is off by > ~3.45e-4; ours is fp32 softmax."""
    params, x, _, _ = make_case(64)
    net = ga3c.Network("gpu:0", "t", 6, max_batch=64)
    net.set_variables(params)
    p, v = net.predict_p_and_v(x)
    assert p.dtype == np.float32 and v.dtype == np.float32 and p.shape == (64, 6) and v.shape == (64,)
    assert np.abs(p.astype(np.float64).sum(axis=1) - 1).max() < 1e-6
    rs = np.random.RandomState(0)
    for i in range(64):
        rs.choice(6, p=p[i])               # raises ValueError if the row is not a distribution


def test_sampling_flip_rate_vs_fp64_oracle(ga3c):
    """Same uniforms, p from the CUDA bf16 trunk vs p from the fp64 oracle: the sampled action differs
    only when u lands within |dp| of a CDF edge (SURVEY A.6)."""
    params, x, _, _ = make_case(256, seed=21)
    net = ga3c.Network("gpu:0", "t", 6, max_batch=256)
    net.set_variables(params)
    p, _ = net.predict_p_and_v(x)
    p64, _ = onp.forward(params, x)
    pq, _ = onp.forward(params, x, quant="bf16")
    u = np.random.default_rng(5).random(256)
    assert np.array_equal(onp.select_actions(p, u), onp.select_actions(pq.astype(np.float32), u))
    flips = int((onp.select_actions(p, u) != onp.select_actions(p64, u)).sum())
    assert flips <= 6, flips               # expected ~ A * |dp| * B ~ 6 * 2e-3 * 256 = 3


# ------------------------------------------------------------------------------------------------
def test_train_step_weights_and_slots(ga3c):
    params, x, y_r, a = make_case(48, seed=2)
    net = ga3c.Network("gpu:0", "t", 6, max_batch=64)
    net.set_variables(params)
    net.learning_rate, net.beta = 3e-4, 0.01
    ms, mom = onp.rmsprop_init(params)
    l_ref, g_ref, p2, ms2, _ = onp.train_step(params, ms, mom, x, y_r.astype(np.float64), a, lr=3e-4, beta=0.01,
                                              quant="bf16")
    losses = net.train(x, y_r.astype(np.float64), a, None, None, 0, fetch_losses=True)   # y_r arrives fp64 (A11)
    assert abs(losses["cost_all"] - l_ref["cost_all"]) <= TOL_LOSS_REL * abs(l_ref["cost_all"])
    got = net.get_variables()
    got_ms, got_mom = net.get_slots()
    for k in got:
        assert np.abs(got[k] - p2[k]).max() <= TOL_W_ABS, k
        assert err(got_ms[k] - 0.99, ms2[k] - 0.99)[1] <= 2 * TOL_GRAD_REL, k     # ms = .99 + .01 g^2
        assert not np.array_equal(got[k], params[k]), k                            # every variable moved
        assert np.all(got_mom[k] == 0), k                                          # mu = 0: slot untouched
    assert net.get_global_step() == 1


def test_rmsprop_kernel_alone_is_fp32_exact(ga3c):
    """ga3c_apply_rmsprop on injected gradients vs the fp32 numpy formula (A.5): <= 1 ulp."""
    import ctypes as C
    import torch
    from ga3c_b200 import _capi
    params, _, _, _ = make_case(1)
    class Cfg(ga3c.Config):
        RMSPROP_MOMENTUM = 0.5
    net = ga3c.Network("gpu:0", "t", 6, max_batch=16, config=Cfg)
    net.set_variables(params)
    rng = np.random.default_rng(0)
    n = net._arena_floats
    g = (rng.standard_normal(n) * 3).astype(np.float32)
    ms0 = rng.uniform(0.5, 2, n).astype(np.float32)
    mom0 = (rng.standard_normal(n) * 1e-3).astype(np.float32)
    w0 = net._download(0)
    for which, arr in ((1, g), (2, ms0), (3, mom0)):
        net._upload(which, arr)
    _capi.check(net._lib.ga3c_apply_rmsprop(net._h, C.c_float(1e-3), None), "rmsprop")
    torch.cuda.synchronize()
    f = np.float32
    ms1 = f(0.99) * ms0 + (f(1) - f(0.99)) * g * g
    mom1 = f(0.5) * mom0 + f(1e-3) * g / np.sqrt(ms1 + f(0.1))
    w1 = w0 - mom1
    assert np.allclose(net._download(2), ms1, rtol=3e-7, atol=0)
    assert np.allclose(net._download(3), mom1, rtol=1e-6, atol=1e-9)      # FMA contraction of the two terms
    assert np.allclose(net._download(0), w1, rtol=0, atol=1e-7)
    # the bf16 shadow of dense1/w follows the update: the next forward uses the new weights
    off, shape = net._table["dense1/w:0"]
    x = onp.synth_frames(rng, 4)
    p, v = net.predict_p_and_v(x)
    pr, vr = onp.forward(net.get_variables(), x, quant="bf16")
    assert np.abs(p - pr).max() <= TOL_P and np.abs(v - vr).max() <= TOL_V


def test_five_step_trajectory(ga3c):
    """Five consecutive train steps on fresh batches track the oracle's trajectory."""
    rng = np.random.default_rng(77)
    params = onp.init_params(rng, 6)
    net = ga3c.Network("gpu:0", "t", 6, max_batch=32)
    net.set_variables(params)
    ms, mom = onp.rmsprop_init(params)
    ref = params
    for step in range(5):
        x = onp.synth_frames(rng, 16)
        y_r, a = onp.synth_targets(rng, 16)
        net.train(x, y_r, a, x, np.zeros(16, bool), 0)
        _, _, ref, ms, mom = onp.train_step(ref, ms, mom, x, y_r, a, lr=net.learning_rate, beta=net.beta, quant="bf16")
        ref = {k: v.astype(np.float32) for k, v in ref.items()}
    got = net.get_variables()
    for k in got:
        assert np.abs(got[k] - ref[k]).max() <= 5 * TOL_W_ABS, k
    assert net.get_global_step() == 5


def test_learning_rate_and_beta_are_read_per_call(ga3c):
    """Server.py:174-175 rewrites model.learning_rate / model.beta while training runs."""
    params, x, y_r, a = make_case(8)
    net = ga3c.Network("gpu:0", "t", 6, max_batch=16)
    net.set_variables(params)
    net.learning_rate = 0.0
    net.train(x, y_r, a, None, None, 0)
    w = net.get_variables()
    assert all(np.array_equal(w[k], params[k]) for k in w)          # lr = 0: weights untouched
    net.beta = 0.5
    l = net.losses(x, y_r, a)
    lr_ = onp.loss_and_grads(params, x, y_r, a, beta=0.5, quant="bf16")[0]
    assert abs(l["cost_p_2"] - lr_["cost_p_2"]) <= TOL_LOSS_REL * abs(lr_["cost_p_2"])


# ------------------------------------------------------------------------------------------------
# size-independent properties at BASELINE.json's full sizes
def test_predict_batch_4096_is_row_independent(ga3c):
    """Config 2's largest batch: predictions are deterministic (same batch twice -> identical bits), every
    row of a 4096-batch equals the same frame predicted in a batch of 128 up to fp32 reassociation (the
    dense1 split-K factor depends on the batch size, like any GEMM library's algorithm choice), and a
    sample of rows matches the oracle."""
    rng = np.random.default_rng(4096)
    params = onp.init_params(rng, 6)
    x = onp.synth_frames(rng, 4096)
    net = ga3c.Network("gpu:0", "t", 6, max_batch=4096)
    net.set_variables(params)
    p, v = net.predict_p_and_v(x)
    p_again, v_again = net.predict_p_and_v(x)
    assert np.array_equal(p, p_again) and np.array_equal(v, v_again)
    for lo in (0, 1920, 3968):
        p2, v2 = net.predict_p_and_v(x[lo:lo + 128])
        assert np.abs(p[lo:lo + 128] - p2).max() <= 1e-6 and np.abs(v[lo:lo + 128] - v2).max() <= 1e-5
    idx = rng.choice(4096, 24, replace=False)
    pr, vr = onp.forward(params, x[idx], quant="bf16")
    assert np.abs(p[idx] - pr).max() <= TOL_P and np.abs(v[idx] - vr).max() <= TOL_V


def test_gradients_are_additive_over_batch_shards_b1024(ga3c):
    """Config 3 (B=1024): every loss term is a SUM over the batch (NetworkVP_discrate.py:61,:83-85), so
    grad(full batch) = sum of grad(shards) -- the identity the data-parallel allreduce relies on."""
    params, x, y_r, a = make_case(1024, seed=8)
    net = ga3c.Network("gpu:0", "t", 6, max_batch=1024)
    net.set_variables(params)
    full_l = net.losses(x, y_r, a)
    full = net.get_gradients()
    acc = {k: np.zeros_like(v, dtype=np.float64) for k, v in full.items()}
    acc_l = 0.0
    for lo in range(0, 1024, 128):
        acc_l += net.losses(x[lo:lo + 128], y_r[lo:lo + 128], a[lo:lo + 128])["cost_all"]
        for k, v in net.get_gradients().items():
            acc[k] += v
    assert abs(acc_l - full_l["cost_all"]) <= 1e-5 * abs(full_l["cost_all"])
    for k in full:
        assert err(full[k], acc[k])[1] <= 2e-4, k      # fp32 accumulation order only
    # and a 64-row shard against the oracle
    _, g_ref = onp.loss_and_grads(params, x[:64], y_r[:64], a[:64], quant="bf16")
    net.losses(x[:64], y_r[:64], a[:64])
    got = net.get_gradients()
    for k in got:
        assert err(got[k], g_ref[k])[1] <= TOL_GRAD_REL, k


def test_train_step_is_bit_reproducible_b1024(ga3c):
    """Weight / bias gradients are per-CTA partial sums added in a fixed order (grad_reduce), the dense1 split-K
    partials likewise: the same batch twice gives identical gradient and loss BITS, also with a different batch
    (other slab contents, other grids) in between."""
    params, x, y_r, a = make_case(1024, seed=21)
    net = ga3c.Network("gpu:0", "t", 6, max_batch=1024)
    net.set_variables(params)
    l0 = net.losses(x, y_r, a)
    g0 = net.get_gradients()
    net.losses(x[:37], y_r[:37], a[:37])
    l1 = net.losses(x, y_r, a)
    g1 = net.get_gradients()
    assert l0 == l1
    for k in g0:
        assert np.array_equal(g0[k], g1[k]), k


def test_uint8_frames_match_normalised_fp32_bit_for_bit(ga3c):
    """F2 ingestion (SURVEY 8f): uint8 pixels k handed over as they are, x = k/128 - 1 (Environment.py:60) applied in the
    kernels' fp32 -> bf16 conversion.  The normalisation is exact, so predictions, losses, gradients and the updated
    weights equal the fp32 path on the normalised frames bit for bit (and therefore match the oracle as it does)."""
    rng = np.random.default_rng(77)
    params = onp.init_params(rng, 6)
    b = 37
    k = rng.integers(0, 256, size=(b, 84 * 84 * 4), dtype=np.uint8)
    x = k.astype(np.float32) / 128.0 - 1.0
    y_r, a = onp.synth_targets(rng, b)
    nets = []
    for frames in (x, k):
        net = ga3c.Network("gpu:0", "t", 6, max_batch=64)
        net.set_variables(params)
        p, v = net.predict_p_and_v(frames)
        l = net.losses(frames, y_r, a)
        g = net.get_gradients()
        net.train(frames, y_r, a, None, None, 0)
        nets.append((p, v, l, g, net.get_variables()))
    (p0, v0, l0, g0, w0), (p1, v1, l1, g1, w1) = nets
    assert np.array_equal(p0, p1) and np.array_equal(v0, v1) and l0 == l1
    for name in g0:
        assert np.array_equal(g0[name], g1[name]), name
        assert np.array_equal(w0[name], w1[name]), name
    pr, vr = onp.forward(params, x, quant="bf16")
    assert np.abs(p1 - pr).max() <= TOL_P and np.abs(v1 - vr).max() <= TOL_V


def test_workspace_grows_for_unbounded_train_batches(ga3c):
    """ThreadTrainer concatenates agent batches without bound (ThreadTrainer.py:48-59)."""
    params, x, y_r, a = make_case(40)
    net = ga3c.Network("gpu:0", "t", 6, max_batch=16)
    net.set_variables(params)
    p, v = net.predict_p_and_v(x)
    pr, vr = onp.forward(params, x, quant="bf16")
    assert np.abs(p - pr).max() <= TOL_P and np.abs(v - vr).max() <= TOL_V
    assert net.train(x, y_r, a, None, None, 0) is None


# ------------------------------------------------------------------------------------------------
# returns and sampling: bit-exact against outputs of the REAL reference (tests/golden)
def test_returns_golden_bit_exact_on_device(ga3c, golden_dir):
    from ga3c_b200.agent_ops import accumulate_rewards
    cases = json.load(open(os.path.join(golden_dir, "returns.json")))
    by_cfg = {}
    for c in cases:
        f = c["flags"]
        by_cfg.setdefault((f["DISCOUNTING"], f["USE_INTERMEDIATE_REWARD"], f["REWARD_CLIPPING"], c["gamma"]), []).append(c)
    for (disc, inter, clip, gamma), group in by_cfg.items():
        class Cfg(ga3c.Config):
            DISCOUNTING, USE_INTERMEDIATE_REWARD, REWARD_CLIPPING = disc, inter, clip
        outs = accumulate_rewards([c["rewards"] for c in group], gamma, [c["terminal"] for c in group], config=Cfg)
        for c, o in zip(group, outs):
            assert [float(r).hex() for r in o] == c["out"]


def test_returns_ragged_and_empty_segments(ga3c):
    from ga3c_b200.agent_ops import accumulate_rewards
    rng = np.random.default_rng(3)
    lens = [0, 1, 2, 5, 0, 1000, 6, 1]               # TIME_MAX upstream 5, fork 1000
    segs = [list(rng.uniform(-2, 2, n)) for n in lens]
    term = [s[-1] if s else 0.0 for s in segs]
    outs = accumulate_rewards(segs, 0.99, term)
    for s, t, o in zip(segs, term, outs):
        assert list(o) == onp.accumulate_rewards(s, 0.99, t)
    outs = accumulate_rewards(segs, 0.99, term, nstep=True)
    for s, t, o in zip(segs, term, outs):
        assert list(o[:-1]) == onp.nstep_returns(s, 0.99, t) if s else len(o) == 0
    assert accumulate_rewards([], 0.99, []) == []


def test_returns_256_agents_t1000(ga3c):
    """SURVEY 8d returns-kernel input: 256 agents x T=1000, closed form R_t = gamma^(n-1-t) r_last."""
    from ga3c_b200.agent_ops import accumulate_rewards
    rng = np.random.default_rng(9)
    segs = [list(rng.uniform(-1, 1, 1000)) for _ in range(256)]
    outs = accumulate_rewards(segs, 0.99, [s[-1] for s in segs])
    for i in (0, 100, 255):
        assert list(outs[i]) == onp.accumulate_rewards(segs[i], 0.99, segs[i][-1])


def test_sampling_golden_bit_exact_on_device(ga3c, golden_dir):
    from ga3c_b200.agent_ops import select_actions
    g = np.load(os.path.join(golden_dir, "sampling.npz"))
    assert np.array_equal(select_actions(g["p"], g["u"]), g["chosen"])
    assert select_actions(np.zeros((0, 6), np.float32), np.zeros(0)).shape == (0,)
    # CDF-edge cases: u exactly on an edge goes right (side='right'); last bin closed by cdf[-1] = 1
    p = np.array([[0.25, 0.25, 0.5], [0.5, 0.5, 0.0], [1.0, 0.0, 0.0]], dtype=np.float32)
    u = np.array([0.25, 0.5, 0.999999], dtype=np.float64)
    assert np.array_equal(select_actions(p, u), onp.select_actions(p, u))


# ------------------------------------------------------------------------------------------------
# the reference's thread / queue contracts on top of the CUDA Network
class _Agent:
    def __init__(self):
        self.wait_q = queue.Queue(maxsize=1)


class _Server:
    def __init__(self, model, n_agents):
        self.model = model
        self.agents = [_Agent() for _ in range(n_agents)]
        self.training_q = queue.Queue(maxsize=100)
        self.trained = []

    def train_model(self, x_, r_, a_, x2_, done_, trainer_id):       # Server.py:141-150
        self.model.train(x_, r_, a_, x2_, done_, trainer_id)
        self.trained.append(x_.shape[0])


def test_predictor_and_trainer_threads_queue_contract(ga3c):
    params, x, y_r, a = make_case(40, seed=5)
    net = ga3c.Network("gpu:0", "t", 6, max_batch=128)
    net.set_variables(params)
    srv = _Server(net, 40)
    pq = queue.Queue(maxsize=100)
    pred = ga3c.ThreadPredictor(srv, 0, onp.STATE_DIM, pq)
    pred.start()
    for i in range(40):
        pq.put((i, x[i]))                                  # ProcessAgent.py:104
    pr, vr = onp.forward(params, x, quant="bf16")
    for i in range(40):
        p_i, v_i = srv.agents[i].wait_q.get(timeout=60)   # ProcessAgent.py:106
        assert p_i.shape == (6,) and np.abs(p_i - pr[i]).max() <= TOL_P and abs(v_i - vr[i]) <= TOL_V
    pred.exit_flag = True

    class Cfg(ga3c.Config):
        TRAINING_MIN_BATCH_SIZE = 20
    tr = ga3c.ThreadTrainer(srv, 0, config=Cfg)
    tr.start()
    for lo in range(0, 40, 8):                             # ProcessAgent.py:175 items (x_, r_, a_, x2_, done_)
        sl = slice(lo, lo + 8)
        srv.training_q.put((x[sl], y_r[sl].astype(np.float64), a[sl], x[sl], np.zeros(8, bool)))
    import time
    t0 = time.time()
    while sum(srv.trained) < 24 and time.time() - t0 < 60:
        time.sleep(0.01)
    tr.exit_flag = True
    assert srv.trained[0] == 24                            # 8+8+8 > 20: first batch that EXCEEDS the minimum
    assert net.get_global_step() >= 1


def test_concurrent_predict_and_train_threads(ga3c):
    """Server.py:123-134: predictors and trainers call into one model concurrently, with no locks."""
    params, x, y_r, a = make_case(32, seed=6)
    net = ga3c.Network("gpu:0", "t", 6, max_batch=32)
    net.set_variables(params)
    net.learning_rate = 0.0                                 # keep weights fixed so predictions are checkable
    pr, vr = onp.forward(params, x, quant="bf16")
    errs = []

    def predictor():
        try:
            for _ in range(30):
                p, v = net.predict_p_and_v(x)
                assert np.abs(p - pr).max() <= TOL_P and np.abs(v - vr).max() <= TOL_V
        except Exception as e:      # noqa
            errs.append(e)

    def trainer():
        try:
            for _ in range(30):
                net.train(x, y_r, a, None, None, 0)
        except Exception as e:      # noqa
            errs.append(e)

    ts = [threading.Thread(target=f) for f in (predictor, predictor, trainer, trainer)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    assert not errs, errs
    assert net.get_global_step() == 60


def test_two_trainer_threads_with_their_own_staging_slots(ga3c):
    """Config.TRAINERS = 2 ThreadTrainers call train concurrently (ThreadTrainer.py:42-62): each trainer_id stages its batch in
    its own slot on its own copy stream, the steps themselves are serialised.  With both threads feeding the SAME batch the
    result cannot depend on the interleaving: it must equal 2 x 6 sequential steps, bit for bit -- a copy racing a step that
    still reads the slot would show up as different weights."""
    params, x, y_r, a = make_case(96, seed=8)
    pageable = (np.array(x, copy=True), np.array(y_r, dtype=np.float64), np.array(a, copy=True))   # y_r as float64 (ProcessAgent.py:99)
    nets = []
    for threads in (1, 2):
        net = ga3c.Network("gpu:0", f"slots{threads}", 6, max_batch=96)
        net.set_variables(params)
        errs = []

        def trainer(tid, steps):
            try:
                for i in range(steps):
                    net.train(*(pageable if i % 2 else (x, y_r, a)), None, None, tid)
            except Exception as e:      # noqa
                errs.append(e)

        if threads == 1:
            trainer(0, 12)
        else:
            ts = [threading.Thread(target=trainer, args=(tid, 6)) for tid in (0, 1)]
            [t.start() for t in ts]
            [t.join() for t in ts]
        assert not errs, errs
        assert net.get_global_step() == 12
        nets.append(net)
    w1, w2 = nets[0].get_variables(), nets[1].get_variables()
    assert all(np.array_equal(w1[k], w2[k]) for k in w1)
    (ms1, _), (ms2, _) = nets[0].get_slots(), nets[1].get_slots()
    assert all(np.array_equal(ms1[k], ms2[k]) for k in ms1)


# ------------------------------------------------------------------------------------------------
def test_checkpoint_round_trip(ga3c, tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    params, x, y_r, a = make_case(8)
    net = ga3c.Network("gpu:0", "ckpt", 6, max_batch=16)
    net.set_variables(params)
    net.train(x, y_r, a, None, None, 0)
    net.save(42)
    want = net.get_variables()
    want_ms, _ = net.get_slots()
    net2 = ga3c.Network("gpu:0", "ckpt", 6, max_batch=16)
    assert net2.load() == 42
    got = net2.get_variables()
    got_ms, _ = net2.get_slots()
    assert all(np.array_equal(got[k], want[k]) and np.array_equal(got_ms[k], want_ms[k]) for k in want)
    assert net2.get_global_step() == 1
    p1, v1 = net.predict_p_and_v(x)
    p2, v2 = net2.predict_p_and_v(x)
    assert np.array_equal(p1, p2) and np.array_equal(v1, v2)


def test_variable_introspection(ga3c):
    net = ga3c.Network("gpu:0", "t", 6, max_batch=16, seed=1)
    assert net.get_variables_names() == list(onp.PARAM_NAMES)          # TF creation order
    shapes = onp.param_shapes(6)
    for k in onp.PARAM_NAMES:
        v = net.get_variable_value(k)
        assert v.shape == shapes[k] and v.dtype == np.float32
    w = net.get_variable_value("dense1/w:0")
    assert np.abs(w).max() <= 1 / np.sqrt(3872) and w.std() > 0         # U(+-1/sqrt(fan_in))
    assert net.get_global_step() == 0


def test_errors_are_raised_not_swallowed(ga3c):
    from ga3c_b200 import _capi
    import ctypes as C
    net = ga3c.Network("gpu:0", "t", 6, max_batch=16)
    with pytest.raises(ValueError):
        net.predict_p_and_v(np.zeros((2, 100), np.float32))
    with pytest.raises(ValueError):
        ga3c.Network("gpu:0", "t", 6, state_dim=4)
    with pytest.raises(ValueError):
        ga3c.Network("cpu:0", "t", 6)
    with pytest.raises(_capi.Ga3cError):
        ga3c.Network("gpu:0", "t", 19)                      # num_actions out of range
    rc = net._lib.ga3c_predict(net._h, None, 4, None, None, None)
    assert rc != 0 and b"null buffer" in net._lib.ga3c_last_error()
    rc = net._lib.ga3c_predict(net._h, C.c_void_p(1), 10 ** 6, C.c_void_p(1), C.c_void_p(1), None)
    assert rc != 0 and b"batch" in net._lib.ga3c_last_error()
    p, v = net.predict_p_and_v(np.zeros((0, onp.STATE_DIM), np.float32))
    assert p.shape == (0, 6) and v.shape == (0,)


# ------------------------------------------------------------------------------------------------
def test_data_parallel_two_gpus_matches_concatenated_batch(ga3c):
    """SURVEY 8e: two ranks (one per GPU, NCCL) on row shards of one global batch == the oracle's single
    step on the concatenated batch, and the replicas stay bit-identical.  Needs >= 2 visible GPUs."""
    import subprocess, sys, torch
    from conftest import ROOT
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs (covered on CPU by tests/test_dataparallel.py with gloo)")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29611", os.path.join(ROOT, "tests", "dp_check_torchrun.py")],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "DP_CHECK OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


@pytest.mark.parametrize("world", [2, 4, 8])
def test_dp_check_oracle_leg_passes_at_every_world_size(ga3c, world):
    """bench.py's dp_check compares an N-rank run at 64 rows per rank with the oracle's steps on the concatenated batch.  A single
    trainer on those concatenated rows (same seeded data, tools/dp_check_proxy.py) reproduces the N-rank distance from the
    oracle to the last digit, so this is the check the driver's scaling run will meet at N = 2, 4, 8 -- including N = 4, where
    one ReLU-gate flip (2.8e-5 in one entry of dense1/b) broke the first, rows-proportional tolerance."""
    import importlib.util
    from conftest import ROOT
    spec = importlib.util.spec_from_file_location("dp_check_proxy", os.path.join(ROOT, "tools", "dp_check_proxy.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    rep = mod.leg(world)
    assert rep["ok"], rep
    assert rep["max_abs_vs_oracle"] < 5e-5 and rep["entries_beyond_1e5"] < 100, rep      # far from what a broken exchange gives
