"""GPU parity tests (`-m gpu`) of the config-4 MLP networks (SURVEY 8a rows A6 / A7): the CUDA path, called through the
C-ABI library (ga3c_mlp_*), against oracle/oracle_mlp.py on the same seeded inputs.

Both sides compute in floating point from fp32 inputs; the CUDA path is fp32 throughout (FMA accumulation, expf / logf /
atan2f), the oracle fp64.  Tolerances (calibrated on B200, frozen here):
    p, v                    |d| <= 2e-5   (v sums 64 products of O(1) terms)
    loss sums               rel <= 2e-5 of sum |terms| (cancellation-safe: compared against the batch size scale)
    gradients               |d| <= 2e-4 * max|ref| per tensor  (batch sums of up to 65,536 fp32 terms, fixed order)
    weights after RMSProp   |d| <= 1e-6   (lr 3e-4 scales the gradient error)
Gradient-less variables of NetworkVP_discrate stay bit-identical.  Two runs of the same step are bit-identical.
The fork NetworkVP's inputs keep its angle head away from the singular point of atan2, where no fp32 implementation can meet
these bounds (_parity.make_mlp_case).  No shape of SHAPES needs a wider bound: at the widest (state_dim 256, 256-term sums)
|dv| <= 5.5e-7 and the gradients stay within 3e-5 relative (B200).
"""
import re

import numpy as np
import pytest

from oracle import oracle_mlp as om
from _parity import err, make_mlp_case, make_mlp_net, near_angle_singularity

pytestmark = pytest.mark.gpu

TOL_PV = 2e-5
TOL_GRAD_REL = 2e-4
TOL_W_ABS = 1e-6

CASES = [("fork_vp", 3, 1), ("fork_vp", 4, 2), ("discrate", 4, 2)]

# The range ga3c_mlp_create accepts (state_dim 1..256, num_actions 1..18, up to 8 DENSE_LAYERS of width 1..256, the last <= 128):
# (kind, state_dim, num_actions, DENSE_LAYERS), the last entry read by 'discrate' only.  The head matrix has n_out = 1 + 2A
# (fork_vp) or 1 + A (discrate) columns; state_dim picks the 16- or 4-byte weight staging of the first layer and, for fork_vp,
# whether the tensor-core path streams its narrow ends (state_dim <= 4, one action).
D = om.DISCRATE_DENSE_LAYERS
SHAPES = [
    ("fork_vp", 1, 1, D),                 # smallest state
    ("fork_vp", 2, 1, D),                 # MountainCarContinuous; still streamed on the tensor-core path
    ("fork_vp", 5, 1, D),                 # one action, state_dim > 4: not streamed; tile-kernel layer-0 dW next to mlp_heads_wgrad
    ("fork_vp", 8, 2, D),                 # LunarLanderContinuous
    ("fork_vp", 24, 4, D),                # BipedalWalker
    ("fork_vp", 256, 18, D),              # largest state; n_out = 37 = MLP_MAX_OUT
    ("discrate", 2, 3, D),                # MountainCar
    ("discrate", 6, 3, D),                # Acrobot
    ("discrate", 8, 4, (64,)),            # LunarLander
    ("discrate", 1, 1, (1,)),             # one action, one hidden unit
    ("discrate", 17, 18, (33,)),          # odd widths: 4-byte staging; n_out = 19
    ("discrate", 64, 2, (16,)),           # widths on the 16-byte staging path
    ("discrate", 256, 5, (256, 128)),     # largest state, largest last width, a 256-wide gradient-less layer in the arena
]


def shape_params(entries):
    """pytest params (kind, s, a, dense) named kind-s-a, plus the widths where DENSE_LAYERS is not the default."""
    out = []
    for kind, s, a, *dense in entries:
        dense = tuple(dense[0]) if dense else D
        name = f"{kind}-{s}-{a}" + ("" if dense == D else "-" + "x".join(map(str, dense)))
        out.append(pytest.param(kind, s, a, dense, id=name))
    return out


ALL_SHAPES = shape_params(CASES + SHAPES)


def config(mlp, dense=D, **knobs):
    """A Config with DENSE_LAYERS = dense and the given knobs, as a user's Config.py would set them."""
    return type("Cfg", (mlp._DefaultConfig,), dict(DENSE_LAYERS=tuple(dense), **knobs))


def tile_switch(num_sms):
    """The smallest batch the fused kernel runs with 64-row tiles: mlp_tile_rows switches from 16-row tiles once
    ceil(B / 64) * 2 >= num_SMs (B = 4,673 on 148 SMs)."""
    return ((num_sms + 1) // 2 - 1) * 64 + 1


def rows(batch, num_sms):
    """A batch parameter: a row count, or 'tile_switch' / 'tile_switch-1' for the two sides of the tile switch."""
    return {"tile_switch": tile_switch(num_sms), "tile_switch-1": tile_switch(num_sms) - 1}.get(batch, batch)


@pytest.fixture(scope="module")
def mlp():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; there is no CPU fallback")
    from ga3c_b200 import mlp_network
    return mlp_network


@pytest.fixture(scope="module")
def num_sms(mlp):
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def test_variable_table_matches_reference_graph(mlp):
    for p in ALL_SHAPES:
        kind, s, a, dense = p.values
        net = make_mlp_net(mlp, kind, s, a, config=config(mlp, dense))
        shapes = om.param_shapes(kind, s, a, dense)
        assert net.get_variables_names() == list(shapes)
        for k, shp in shapes.items():
            assert net.get_variable_value(k).shape == tuple(shp)
        assert set(net.get_variables_names()) - set(net.live_variables()) == set(om.dead_params(kind, dense))
        v = net.get_variables()
        assert all(np.abs(t).max() <= 0.3 for t in v.values())          # U(-0.3, 0.3), NetworkVP.py:199-202


@pytest.mark.parametrize("kind,s,a,dense", ALL_SHAPES)
@pytest.mark.parametrize("batch", [1, 5, 63, 64, 65, 128, 1000, "tile_switch", 5000])
def test_predict_matches_oracle(mlp, num_sms, kind, s, a, dense, batch):
    """16-row tiles up to the tile switch, 64-row tiles from it on (fork_vp with one action and state_dim <= 4 takes the streamed
    tensor-core path from 4,096 rows on)."""
    batch = rows(batch, num_sms)
    params, x, _, _ = make_mlp_case(kind, s, a, batch, dense_layers=dense)
    net = make_mlp_net(mlp, kind, s, a, config=config(mlp, dense))
    net.set_variables(params)
    p, v = net.predict_p_and_v(x)
    p_ref, v_ref = om.forward(params, x, kind, dense_layers=dense)
    assert p.shape == (batch, a) and v.shape == (batch,) and p.dtype == np.float32
    assert err(p, p_ref)[0] <= TOL_PV and err(v, v_ref)[0] <= TOL_PV, (err(p, p_ref), err(v, v_ref))


@pytest.mark.parametrize("kind,s,a,dense", ALL_SHAPES)
@pytest.mark.parametrize("batch", [1, 7, 64, 200, 1024, "tile_switch-1", "tile_switch", 5000])
def test_losses_and_gradients_match_oracle(mlp, num_sms, kind, s, a, dense, batch):
    """fork_vp takes the tensor-core path from 4,096 rows on: streamed narrow ends for one action and state_dim <= 4, the fused
    kernel's phases otherwise."""
    batch = rows(batch, num_sms)
    params, x, y_r, act = make_mlp_case(kind, s, a, batch, seed=7, dense_layers=dense)
    net = make_mlp_net(mlp, kind, s, a, config=config(mlp, dense))
    net.set_variables(params)
    net.beta = 0.01
    losses = net.losses(x, y_r, act)
    losses_ref, grads_ref = om.loss_and_grads(params, x, y_r, act, kind, beta=0.01, dense_layers=dense)
    for k in ("cost_p_1", "cost_p_2", "cost_v", "cost_all"):
        assert abs(losses[k] - losses_ref[k]) <= 2e-5 * max(batch, abs(losses_ref[k])), (k, losses[k], losses_ref[k])
    grads = net.get_gradients()
    assert set(grads) == set(grads_ref)
    for k, g_ref in grads_ref.items():
        d, r = err(grads[k], g_ref)
        assert r <= TOL_GRAD_REL or d <= 1e-6, (k, d, r)


@pytest.mark.parametrize("kind,s,a", [("fork_vp", 3, 1), ("discrate", 4, 2)])
def test_golden_fixture(mlp, kind, s, a, golden_dir):
    """The committed fixture tests/golden/mlp_b6.npz (torch-autograd restatement, oracle/gen_golden.py: gen_mlp)."""
    import os
    g = np.load(os.path.join(golden_dir, "mlp_b6.npz"))
    params = om.init_params(np.random.default_rng(2024), kind, s, a)            # as oracle/gen_golden.py: gen_mlp drew them
    grads_ref = {k[len(kind) + 6:]: g[k] for k in g.files if k.startswith(kind + "_grad_")}
    x, y_r, act = g[kind + "_x"], g[kind + "_yr"], g[kind + "_a"]
    net = make_mlp_net(mlp, kind, s, a)
    net.set_variables(params)
    net.beta = 0.01
    p, v = net.predict_p_and_v(x)
    assert err(p, g[kind + "_p"])[0] <= TOL_PV and err(v, g[kind + "_v"])[0] <= TOL_PV
    l = net.losses(x, y_r, act)
    got = np.array([l[k] for k in ("cost_p_1", "cost_p_2", "cost_p", "cost_v", "cost_all")])
    assert np.abs(got - g[kind + "_losses"]).max() <= 2e-5 * x.shape[0]
    grads = net.get_gradients()
    assert set(grads) == set(grads_ref)
    for k, g_ref in grads_ref.items():
        d, r = err(grads[k], g_ref)
        assert r <= TOL_GRAD_REL or d <= 1e-6, (k, d, r)


def test_min_policy_mix(mlp):
    """MIN_POLICY > 0 (NetworkVP_discrate.py:69-71): p = (softmax + m) / (1 + m A)."""
    class Cfg(mlp._DefaultConfig):
        MIN_POLICY = 0.05
    kind, s, a, b = "discrate", 4, 2, 300
    params, x, y_r, act = make_mlp_case(kind, s, a, b, seed=3)
    net = make_mlp_net(mlp, kind, s, a, config=Cfg)
    net.set_variables(params)
    p, v = net.predict_p_and_v(x)
    p_ref, v_ref = om.forward(params, x, kind, min_policy=0.05)
    assert err(p, p_ref)[0] <= TOL_PV
    losses = net.losses(x, y_r, act)
    losses_ref, grads_ref = om.loss_and_grads(params, x, y_r, act, kind, beta=0.01, min_policy=0.05)
    assert abs(losses["cost_all"] - losses_ref["cost_all"]) <= 2e-5 * b
    grads = net.get_gradients()
    for k, g_ref in grads_ref.items():
        assert err(grads[k], g_ref)[1] <= TOL_GRAD_REL, k


def test_log_softmax_knob(mlp):
    """Config.USE_LOG_SOFTMAX = True (NetworkVP_discrate.py:64-71): exact log_softmax, no MIN_POLICY mix, no epsilon floor."""
    class Cfg(mlp._DefaultConfig):
        USE_LOG_SOFTMAX = True
        MIN_POLICY = 0.05                  # ignored by this branch
    kind, s, a, b = "discrate", 4, 2, 500
    params, x, y_r, act = make_mlp_case(kind, s, a, b, seed=5)
    net = make_mlp_net(mlp, kind, s, a, config=Cfg)
    net.set_variables(params)
    p, v = net.predict_p_and_v(x)
    p_ref, v_ref = om.forward(params, x, kind, use_log_softmax=True)
    assert err(p, p_ref)[0] <= TOL_PV and err(v, v_ref)[0] <= TOL_PV
    losses = net.losses(x, y_r, act)
    losses_ref, grads_ref = om.loss_and_grads(params, x, y_r, act, kind, beta=0.01, use_log_softmax=True)
    for k in ("cost_p_1", "cost_p_2", "cost_v", "cost_all"):
        assert abs(losses[k] - losses_ref[k]) <= 2e-5 * b, (k, losses[k], losses_ref[k])
    grads = net.get_gradients()
    for k, g_ref in grads_ref.items():
        assert err(grads[k], g_ref)[1] <= TOL_GRAD_REL, (k, err(grads[k], g_ref))


def test_grad_clip_knob(mlp):
    """Config.USE_GRAD_CLIP: the fork's NetworkVP clips per variable and advances global_step (NetworkVP.py:138-141);
    NetworkVP_discrate with its default gradient-less layers cannot build that graph (clip_by_average_norm(None)) and is
    refused; with a single dense layer it clips and leaves global_step alone (NetworkVP_discrate.py:118-121)."""
    clip = 1e-3
    class Cfg(mlp._DefaultConfig):
        USE_GRAD_CLIP = True
        GRAD_CLIP_NORM = clip
    class Cfg1(Cfg):
        DENSE_LAYERS = (10,)
    with pytest.raises(Exception):
        make_mlp_net(mlp, "discrate", 4, 2, config=Cfg)
    for kind, s, a, cfg, steps_counted in (("fork_vp", 3, 1, Cfg, True), ("discrate", 4, 2, Cfg1, False)):
        b = 300
        rng = np.random.default_rng(3)
        net = make_mlp_net(mlp, kind, s, a, config=cfg)
        params = net.get_variables()
        x = rng.uniform(-1, 1, size=(b, s)).astype(np.float32)
        y_r = rng.uniform(-1, 1, size=b).astype(np.float32)
        act = (rng.uniform(-1, 1, size=(b, a)).astype(np.float32) if kind == "fork_vp"
               else np.eye(a, dtype=np.float32)[rng.integers(0, a, size=b)])
        ref_p = {k: v.copy() for k, v in params.items()}
        ref_ms = {k: np.ones_like(v) for k, v in params.items()}
        ref_mom = {k: np.zeros_like(v) for k, v in params.items()}
        for _ in range(2):
            net.train(x, y_r, act, None, None, 0)
            _, grads, ref_p, ref_ms, ref_mom = om.train_step(ref_p, ref_ms, ref_mom, x, y_r, act, kind, lr=3e-4, grad_clip=clip,
                                                             dense_layers=cfg.DENSE_LAYERS)
        _, raw = om.loss_and_grads(params, x, y_r, act, kind, dense_layers=cfg.DENSE_LAYERS)   # un-clipped, initial weights
        avg = [np.sqrt((g.astype(np.float64) ** 2).sum()) / g.size for g in raw.values()]
        assert max(avg) > clip, avg                                     # the threshold is active
        w = net.get_variables()
        for k in w:
            assert err(w[k], ref_p[k])[0] <= TOL_W_ABS, (kind, k, err(w[k], ref_p[k]))
        assert net.get_global_step() == (2 if steps_counted else 0)


@pytest.mark.parametrize("kind,s,a", CASES)
def test_dual_rmsprop_knob(mlp, kind, s, a):
    """Config.DUAL_RMSPROP (NetworkVP.py:107-118, :143-147): two optimizers, semantics as oracle_mlp.train_step_dual."""
    class Cfg(mlp._DefaultConfig):
        DUAL_RMSPROP = True
    b = 400
    params, x, y_r, act = make_mlp_case(kind, s, a, b, seed=29)
    net = make_mlp_net(mlp, kind, s, a, config=Cfg)
    net.set_variables(params)
    ones = {k: np.ones_like(v) for k, v in params.items()}
    zeros = {k: np.zeros_like(v) for k, v in params.items()}
    ref, sp, sv = params, (ones, zeros), (ones, zeros)
    for _ in range(3):
        net.train(x, y_r, act, None, None, 0)
        _, gp, gv, ref, sp, sv = om.train_step_dual(ref, sp, sv, x, y_r, act, kind, lr=3e-4, beta=0.01)
    w = net.get_variables()
    for k in w:
        assert err(w[k], ref[k])[0] <= 2 * TOL_W_ABS, (k, err(w[k], ref[k]))
    ms_p, _ = net.get_slots(0)
    ms_v, _ = net.get_slots(1)
    for k in gp:
        assert err(ms_p[k], sp[0][k])[1] <= 1e-4, k
    for k in gv:
        assert err(ms_v[k], sv[0][k])[1] <= 1e-4, k
    assert np.array_equal(ms_p["logits_v/w:0"], ones["logits_v/w:0"])
    assert net.get_global_step() == 6
    for k in om.dead_params(kind):
        assert np.array_equal(w[k], params[k])


@pytest.mark.parametrize("kind,s,a", CASES)
def test_dual_rmsprop_with_grad_clip(mlp, kind, s, a):
    """Config.DUAL_RMSPROP + USE_GRAD_CLIP (NetworkVP.py:127-137, NetworkVP_discrate.py:107-117): tf.clip_by_norm per variable
    and optimizer; variables without a gradient are filtered (`if not g is None`), so NetworkVP_discrate's gradient-less
    layers are legal here; the fork's NetworkVP passes global_step to both apply_gradients calls, NetworkVP_discrate to none."""
    clip = 2e-2
    class Cfg(mlp._DefaultConfig):
        DUAL_RMSPROP = True
        USE_GRAD_CLIP = True
        GRAD_CLIP_NORM = clip
    b = 400
    params, x, y_r, act = make_mlp_case(kind, s, a, b, seed=37)
    net = make_mlp_net(mlp, kind, s, a, config=Cfg)
    net.set_variables(params)
    ones = {k: np.ones_like(v) for k, v in params.items()}
    zeros = {k: np.zeros_like(v) for k, v in params.items()}
    ref, sp, sv = params, (ones, zeros), (ones, zeros)
    for _ in range(2):
        net.train(x, y_r, act, None, None, 0)
        _, gp, gv, ref, sp, sv = om.train_step_dual(ref, sp, sv, x, y_r, act, kind, lr=3e-4, beta=0.01, grad_clip=clip)
    norms = [float(np.sqrt((g.astype(np.float64) ** 2).sum())) for g in list(gp.values()) + list(gv.values())]
    assert any(v > clip for v in norms), norms                              # the threshold is active
    w = net.get_variables()
    for k in w:
        assert err(w[k], ref[k])[0] <= 2 * TOL_W_ABS, (k, err(w[k], ref[k]))
    assert net.get_global_step() == (4 if kind == "fork_vp" else 0)
    for k in om.dead_params(kind):
        assert np.array_equal(w[k], params[k])


def train_three_steps(mlp, kind, s, a, dense, momentum=0.0):
    """Three opt.minimize steps of the network and of the oracle from the same weights, RMSPROP_MOMENTUM = momentum; the loss of
    every step is checked.  fork_vp: rows that bring an angle near the singular point of the angle head at any step's weights are
    redrawn first (_parity.make_mlp_case).  -> (net, initial params, oracle params, ms, mom)"""
    b = 777
    params, x, y_r, act = make_mlp_case(kind, s, a, b, seed=11, dense_layers=dense)
    rng = np.random.default_rng(11)
    while True:
        ref = [({k: v.copy() for k, v in params.items()}, {k: np.ones_like(v) for k, v in params.items()},
                {k: np.zeros_like(v) for k, v in params.items()})]
        losses_ref = []
        for _ in range(3):
            l, _, *state = om.train_step(*ref[-1], x, y_r, act, kind, lr=3e-4, beta=0.01, mu=momentum, dense_layers=dense)
            losses_ref.append(l)
            ref.append(tuple(state))
        bad = np.zeros(b, bool)
        if kind == "fork_vp":
            for w, _, _ in ref:
                bad |= near_angle_singularity(w, x)
        if not bad.any():
            break
        x[bad] = rng.uniform(-1, 1, size=(int(bad.sum()), s)).astype(np.float32)
    net = make_mlp_net(mlp, kind, s, a, config=config(mlp, dense, RMSPROP_MOMENTUM=momentum))
    net.set_variables(params)
    net.learning_rate, net.beta = 3e-4, 0.01
    for step in range(3):
        got = net.train(x, y_r, act, None, None, 0, fetch_losses=True)
        assert abs(got["cost_all"] - losses_ref[step]["cost_all"]) <= 2e-5 * b, (step, got, losses_ref[step])
    assert net.get_global_step() == 3
    return (net, params) + ref[-1]


@pytest.mark.parametrize("kind,s,a,dense", ALL_SHAPES)
def test_train_steps_match_oracle(mlp, kind, s, a, dense):
    """Three opt.minimize steps: weights, ms slot, global_step; gradient-less variables untouched (bit-identical)."""
    net, params, ref_p, ref_ms, _ = train_three_steps(mlp, kind, s, a, dense)
    w = net.get_variables()
    ms, _ = net.get_slots()
    for k in params:
        assert err(w[k], ref_p[k])[0] <= TOL_W_ABS, (k, err(w[k], ref_p[k]))
        assert err(ms[k], ref_ms[k])[1] <= 1e-4, (k, err(ms[k], ref_ms[k]))
    for k in om.dead_params(kind, dense):
        assert np.array_equal(w[k], params[k]) and np.array_equal(ms[k], np.ones_like(params[k]))


@pytest.mark.parametrize("kind,s,a,dense", shape_params([("fork_vp", 24, 4), ("discrate", 256, 5, (256, 128))]))
def test_momentum_train_steps_match_oracle(mlp, kind, s, a, dense):
    """RMSPROP_MOMENTUM = 0.9: the optimizer's momentum instantiation over the live prefix of the arena.  Weights, ms and mom
    against the oracle; the gradient-less variables (a 256 x 256 layer for discrate) and their slots stay bit-identical."""
    net, params, ref_p, ref_ms, ref_mom = train_three_steps(mlp, kind, s, a, dense, momentum=0.9)
    w = net.get_variables()
    ms, mom = net.get_slots()
    dead = om.dead_params(kind, dense)
    for k in params:
        assert err(w[k], ref_p[k])[0] <= TOL_W_ABS, (k, err(w[k], ref_p[k]))
        assert err(ms[k], ref_ms[k])[1] <= 1e-4, (k, err(ms[k], ref_ms[k]))
        if k not in dead:
            assert np.abs(mom[k]).max() > 0, k
            assert err(mom[k], ref_mom[k])[1] <= 1e-4, (k, err(mom[k], ref_mom[k]))
    assert len(dead) == (2 if kind == "discrate" else 0)
    for k in dead:
        assert np.array_equal(w[k], params[k]), k
        assert np.array_equal(ms[k], np.ones_like(params[k])) and np.array_equal(mom[k], np.zeros_like(params[k])), k


def test_full_size_batch_and_reproducibility(mlp):
    """BASELINE config 4's large batch (65,536): direct parity with the oracle, and bit-identical repeats (fixed-order sums)."""
    kind, s, a, b = "fork_vp", 3, 1, 65536
    params, x, y_r, act = make_mlp_case(kind, s, a, b, seed=21)
    net = make_mlp_net(mlp, kind, s, a, max_batch=b)
    net.set_variables(params)
    p, v = net.predict_p_and_v(x)
    p_ref, v_ref = om.forward(params, x, kind)
    assert err(p, p_ref)[0] <= TOL_PV and err(v, v_ref)[0] <= TOL_PV
    l1 = net.losses(x, y_r, act)
    g1 = net.get_gradients()
    l2 = net.losses(x, y_r, act)
    g2 = net.get_gradients()
    assert l1 == l2 and all(np.array_equal(g1[k], g2[k]) for k in g1)
    losses_ref, grads_ref = om.loss_and_grads(params, x, y_r, act, kind, beta=0.01)
    assert abs(l1["cost_all"] - losses_ref["cost_all"]) <= 2e-5 * b
    for k, g_ref in grads_ref.items():
        assert err(g1[k], g_ref)[1] <= TOL_GRAD_REL, (k, err(g1[k], g_ref))


def check_tensor_cores_against_oracle_and_fp32(mlp, monkeypatch, s, a, batch, tc):
    """fork_vp (s, a) with GA3C_MLP_TC = tc (None: unset, the default 4,096-row threshold) against the oracle and against a
    GA3C_MLP_TC=0 handle (fp32 FMA path): predictions, losses and gradients.  Predict streams (front, 3 GEMMs, heads) only for
    one action and state_dim <= 4; otherwise it is one fused launch."""
    kind = "fork_vp"
    params, x, y_r, act = make_mlp_case(kind, s, a, batch, seed=11)
    out = {}
    for mode in ("1", "0"):
        if mode == "1" and tc is None:
            monkeypatch.delenv("GA3C_MLP_TC", raising=False)
        else:
            monkeypatch.setenv("GA3C_MLP_TC", tc if mode == "1" else "0")   # read at construction: N = tensor cores from N rows, 0 = never
        net = make_mlp_net(mlp, kind, s, a, max_batch=batch)
        net.set_variables(params)
        net.beta = 0.01
        n0 = net.launch_count()
        pv = net.predict_p_and_v(x)
        n1 = net.launch_count()
        out[mode] = (net.losses(x, y_r, act), net.get_gradients(), net.launch_count() - n1, pv, n1 - n0)
    assert out["1"][2] > out["0"][2] == 3, (out["1"][2], out["0"][2])      # the GEMM launches really ran
    streamed = a == 1 and s <= 4
    assert out["0"][4] == 1 and out["1"][4] == (5 if streamed else 1), (out["1"][4], out["0"][4])
    p_ref, v_ref = om.forward(params, x, kind)
    for mode in ("1", "0"):
        p, v = out[mode][3]
        assert err(p, p_ref)[0] <= TOL_PV and err(v, v_ref)[0] <= TOL_PV, (mode, err(p, p_ref), err(v, v_ref))
    losses_ref, grads_ref = om.loss_and_grads(params, x, y_r, act, kind, beta=0.01)
    losses, grads, _, _, _ = out["1"]
    for k in ("cost_p_1", "cost_p_2", "cost_v", "cost_all"):
        assert abs(losses[k] - losses_ref[k]) <= 2e-5 * max(batch, abs(losses_ref[k])), (k, losses[k], losses_ref[k])
    for k, g_ref in grads_ref.items():
        d, r = err(grads[k], g_ref)
        assert r <= TOL_GRAD_REL or d <= 1e-6, (k, d, r)
        d, r = err(grads[k], out["0"][1][k])
        assert r <= TOL_GRAD_REL or d <= 1e-6, ("vs fp32 path", k, d, r)


@pytest.mark.parametrize("s,a", [(3, 1), (4, 2), (5, 1), (8, 2), (24, 4)])
@pytest.mark.parametrize("batch", [33, 128, 1000, 4097])
def test_tensor_core_wide_layers_match_oracle_and_the_fp32_path(mlp, monkeypatch, s, a, batch):
    """The 256 -> 256, 256 -> 100 and 100 -> 64 layers of the fork NetworkVP as 3xTF32 tcgen05 GEMMs (mlp_tc.cu; taken from 4096
    rows on, forced here from 1 row): same tolerances against the oracle as the fp32 FMA path, and close to that path itself --
    predictions, losses and gradients.  With one action and state_dim <= 4 the narrow ends are the streaming kernels of
    mlp_stream.cu; otherwise the fused kernel's phases, and with state_dim > 4 layer 0's weight gradient comes from the tile
    kernel (mlp_wgrad) instead of mlp_skinny_wgrad."""
    check_tensor_cores_against_oracle_and_fp32(mlp, monkeypatch, s, a, batch, tc="1")


def test_tensor_cores_from_the_default_threshold(mlp, monkeypatch):
    """GA3C_MLP_TC unset: a LunarLanderContinuous-sized NetworkVP (8, 2) crosses the default 4,096-row threshold at 5,000 rows."""
    check_tensor_cores_against_oracle_and_fp32(mlp, monkeypatch, 8, 2, 5000, tc=None)


def test_batch_sum_is_additive(mlp):
    """Size-independent property: every loss term and gradient is a SUM over the batch (NetworkVP_discrate.py:61,:83-85), so
    the gradient of a concatenated batch equals the sum of the parts' gradients."""
    kind, s, a = "discrate", 4, 2
    params, x, y_r, act = make_mlp_case(kind, s, a, 3000, seed=31)
    net = make_mlp_net(mlp, kind, s, a)
    net.set_variables(params)
    net.losses(x, y_r, act)
    g_all = net.get_gradients()
    net.losses(x[:1100], y_r[:1100], act[:1100])
    g_a = net.get_gradients()
    net.losses(x[1100:], y_r[1100:], act[1100:])
    g_b = net.get_gradients()
    for k in g_all:
        assert err(g_a[k] + g_b[k], g_all[k])[1] <= 1e-5, k


@pytest.mark.parametrize("kind,s,a,dense", shape_params([("discrate", 17, 18, (33,)), ("discrate", 256, 5, (256, 128)),
                                                        ("fork_vp", 8, 2)]))
def test_rows_do_not_depend_on_the_tile_mode(mlp, num_sms, kind, s, a, dense):
    """Predict rows of a batch run with 64-row tiles equal, bit for bit, the same rows predicted inside a 100-row batch (16-row
    tiles): every output is one thread's FMA chain over k in the same order in both instantiations of the fused kernel.  And
    the gradients at the tile switch equal the sum of those of its two parts, one on each side of the switch."""
    t = tile_switch(num_sms)
    big = max(5000, t)
    params, x, y_r, act = make_mlp_case(kind, s, a, big, seed=41, dense_layers=dense)
    net = make_mlp_net(mlp, kind, s, a, config=config(mlp, dense))
    net.set_variables(params)
    p_big, v_big = net.predict_p_and_v(x)
    pick = np.arange(100) * (big // 100)                   # rows from 100 different 64-row tiles, at varied positions in them
    p_small, v_small = net.predict_p_and_v(x[pick])
    assert np.array_equal(p_small, p_big[pick]) and np.array_equal(v_small, v_big[pick]), \
        (np.abs(p_small - p_big[pick]).max(), np.abs(v_small - v_big[pick]).max())
    net.losses(x[:t], y_r[:t], act[:t])
    g_all = net.get_gradients()
    net.losses(x[:t - 1], y_r[:t - 1], act[:t - 1])
    g_a = net.get_gradients()
    net.losses(x[t - 1:t], y_r[t - 1:t], act[t - 1:t])
    g_b = net.get_gradients()
    for k in g_all:
        assert err(g_a[k] + g_b[k], g_all[k])[1] <= 1e-5, (k, err(g_a[k] + g_b[k], g_all[k]))


def test_errors_and_checkpoint_roundtrip(mlp, tmp_path, monkeypatch):
    net = make_mlp_net(mlp, "fork_vp", 3, 1)
    with pytest.raises(ValueError):
        net.predict_p_and_v(np.zeros((4, 5), np.float32))
    p, v = net.predict_p_and_v(np.zeros((0, 3), np.float32))
    assert p.shape == (0, 1) and v.shape == (0,)
    assert net.train(np.zeros((0, 3), np.float32), np.zeros(0), np.zeros((0, 1)), None, None, 0) is None
    with pytest.raises(Exception):
        make_mlp_net(mlp, "fork_vp", 300, 1)                # state_dim out of range: ga3c_mlp_create fails loudly
    monkeypatch.chdir(tmp_path)
    params, x, y_r, act = make_mlp_case("fork_vp", 3, 1, 50)
    net.train(x, y_r, act, None, None, 0)
    net.save(12)
    other = make_mlp_net(mlp, "fork_vp", 3, 1, seed=99)
    other.model_name = net.model_name
    assert other.load() == 12 and other.get_global_step() == 1
    a, b = net.get_variables(), other.get_variables()
    assert all(np.array_equal(a[k], b[k]) for k in a)
    assert net.launch_count() > 0


@pytest.mark.parametrize("kind,s,a,dense,message", [
    pytest.param("fork_vp", 3, 0, D, "num_actions must be 1..18", id="no-action"),
    pytest.param("discrate", 4, 19, D, "num_actions must be 1..18", id="19-actions"),
    pytest.param("discrate", 4, 2, (10, 129), "the last dense width must be <= 128", id="last-width-129"),
    pytest.param("discrate", 4, 2, (10, 0, 10), "dense widths must be 1..256", id="width-0"),
    pytest.param("discrate", 4, 2, (10,) * 9, "at most 8 entries", id="9-dense-layers"),
    pytest.param("fork_vp", 0, 1, D, "state_dim must be 1..256", id="no-state"),
])
def test_create_refuses_shapes_outside_the_range(mlp, kind, s, a, dense, message):
    """One step past each edge of the range ga3c_mlp_create accepts: an error that says which, and no network."""
    from ga3c_b200 import _capi
    with pytest.raises((ValueError, _capi.Ga3cError), match=re.escape(message)):
        make_mlp_net(mlp, kind, s, a, config=config(mlp, dense))
