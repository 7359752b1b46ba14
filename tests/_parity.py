"""Shared helpers of the GPU parity tests: run the CUDA path and the oracle on the same seeded
inputs and report per-tensor error figures.  The oracle is the checker, never the thing measured."""
from __future__ import annotations

import numpy as np

from oracle import oracle_mlp as om
from oracle import oracle_np as onp


def make_case(batch: int, num_actions: int = 6, seed: int = 12345):
    rng = np.random.default_rng(seed)
    params = onp.init_params(rng, num_actions)
    x = onp.synth_frames(rng, batch)
    y_r, a = onp.synth_targets(rng, batch, num_actions)
    return params, x, y_r, a


def make_mlp_net(mlp, kind: str, s: int, a: int, **kw):
    """The MLP network of `kind` ('fork_vp': NetworkVP, 'discrate': NetworkVP_discrate) for state size s and a actions; kw go to
    the constructor (config=, max_batch=, seed=)."""
    cls = mlp.NetworkVP if kind == "fork_vp" else mlp.NetworkVP_discrate
    return cls("gpu:0", "test" + kind.replace("_", ""), a, s, **kw)   # no "_": the reference parses the episode out of the name


# fork_vp: least distance of (sigmoid(out_x), sigmoid(out_y)) from (0.5, 0.5), where p = atan2(Y, X) / pi is singular
ANGLE_R_MIN = 0.01


def near_angle_singularity(params, x):
    """fork_vp: which rows of x have an angle closer than ANGLE_R_MIN to the singular point of the angle head under `params`."""
    _, _, f = om.forward(params, x, "fork_vp", keep=True)
    return (np.hypot(f["ox"] - 0.5, f["oy"] - 0.5) < ANGLE_R_MIN).any(axis=1)


def make_mlp_case(kind: str, s: int, a: int, b: int, seed: int = 12345, dense_layers=om.DISCRATE_DENSE_LAYERS):
    """Seeded MLP weights (dense_layers = Config.DENSE_LAYERS, 'discrate' only) and b rows of x, y_r and actions.

    fork_vp: rows with an angle closer than ANGLE_R_MIN to the singular point of the angle head are redrawn.  There X = sigmoid(z_x)
    - 0.5 and Y carry the fp32 rounding of sigmoid near 0.5 (delta = 2^-23, one ulp), which p amplifies by up to sqrt(2) / (pi r)
    and the out_x / out_y gradients by 1 / r^2: any fp32 implementation differs from the fp64 oracle there, TF's included.  Measured
    on a B200 for (256, 18) at 5,000 rows, with an angle at r = 7.3e-4: |dp| = 5.55e-5 (the oracle itself run in fp32: 4.5e-5) and
    1.15e-3 relative in logits_p/out_y/w (2.9e-5 with the 42 rows that hold an angle at r < 5e-3 removed).  At r >= ANGLE_R_MIN
    the bound is sqrt(2) 2^-23 / (pi r) <= 5.4e-6 for p, a quarter of the p, v tolerance.  The rows drawn for state_dim 3 and 4
    lie at r > 0.05 and are never redrawn.  Training moves the angles: a test that trains checks them at every step's weights."""
    rng = np.random.default_rng(seed)
    params = om.init_params(rng, kind, s, a, dense_layers)
    x = rng.uniform(-1, 1, size=(b, s)).astype(np.float32)
    y_r = rng.uniform(-1, 1, size=b).astype(np.float32)
    if kind == "fork_vp":
        act = rng.uniform(-1, 1, size=(b, a)).astype(np.float32)      # continuous action (ProcessAgent.py:92-93)
        rows = np.arange(b)
        while rows.size:
            rows = rows[near_angle_singularity(params, x[rows])]
            x[rows] = rng.uniform(-1, 1, size=(rows.size, s)).astype(np.float32)
    else:
        act = np.eye(a, dtype=np.float32)[rng.integers(0, a, size=b)]
    return params, x, y_r, act


def err(got, ref):
    """(max abs error, max abs error / max |ref|)."""
    got = np.asarray(got, dtype=np.float64).ravel()
    ref = np.asarray(ref, dtype=np.float64).ravel()
    d = float(np.abs(got - ref).max()) if got.size else 0.0
    s = float(np.abs(ref).max()) if ref.size else 0.0
    return d, d / max(s, 1e-30)


def layer_report(net, params, x, y_r, a, *, beta=0.01, log_eps=1e-6, min_policy=0.0, use_log_softmax=False):
    """Runs predict + forward_backward on `net` (weights := params) and compares every stored
    activation, every gradient and the loss sums with the bf16-rounding-point oracle (fp64 accumulate).
    Returns {name: (abs_err, rel_err)}."""
    net.set_variables(params)
    net.beta = beta
    rep = {}
    p, v = net.predict_p_and_v(x)
    losses_ref, grads_ref, f = onp.loss_and_grads(params, x, y_r, a, beta=beta, log_eps=log_eps,
                                                  min_policy=min_policy, quant="bf16", keep=True,
                                                  use_log_softmax=use_log_softmax)
    rep["p"] = err(p, f["p"])
    rep["v"] = err(v, f["v"])
    net.keep_dn1(True)          # dn1 is consumed on chip by the fused conv backward; ask for a copy
    losses = net.losses(x, y_r, a)
    net.keep_dn1(False)
    b = x.shape[0]
    rep["n1"] = err(net.workspace(0), f["n1"].reshape(b, -1))
    rep["n2"] = err(net.workspace(1), f["n2"].reshape(b, -1))
    rep["d1"] = err(net.workspace(2), f["d1"])
    rep["dd1"] = err(net.workspace(3), f["dd1"])
    rep["dn2"] = err(net.workspace(4), f["dn2"])
    rep["dn1"] = err(net.workspace(5), f["dn1"])
    # Layer-local view of the two masked data gradients: the same oracle arithmetic applied to the CUDA path's OWN stored inputs
    # (dd1 / dn2 and the activation masks).  A stored activation that sits within an fp32-vs-fp64 accumulation difference of
    # the ReLU boundary flips its mask bit; the global comparison above then shows that element's whole gradient (and what
    # it spreads to upstream) as an error although every kernel did its arithmetic right.  At full-size batches (millions of
    # activations) a handful of such flips is certain; the local view is immune, and `outliers` says how few elements differ.
    w12q = f["w12"]
    n1_mask = (net.workspace(0).reshape(b, -1) > 0)
    n2_mask = (net.workspace(1).reshape(b, -1) > 0)
    dn2_cuda = net.workspace(4).astype(np.float64).reshape(b * onp.H2 * onp.H2, onp.C2_OUT)
    dd1_cuda = net.workspace(3).astype(np.float64).reshape(b, -1)
    dn2_local = onp.bf16_round((dd1_cuda @ f["w1"].T) * n2_mask)
    dn1_local = onp._col2im(dn2_cuda @ w12q.T, b, onp.H1, onp.C2_K, onp.C2_S, onp.P2_LO, onp.P2_HI, onp.H2, onp.C1_OUT)
    dn1_local = onp.bf16_round(dn1_local.reshape(b, -1) * n1_mask)
    rep["dn2_local"] = err(net.workspace(4), dn2_local)
    rep["dn1_local"] = err(net.workspace(5), dn1_local)
    for k in ("dn1", "dn2"):
        got, ref = net.workspace(5 if k == "dn1" else 4).ravel(), np.asarray(f[k], dtype=np.float64).ravel()
        rep[k + "_outliers"] = (float((np.abs(got - ref) > 2.0 ** -7 * np.abs(ref).max()).mean()), 0.0)
    for k in ("cost_p_1", "cost_p_2", "cost_v", "cost_all"):
        rep["loss/" + k] = err([losses[k]], [losses_ref[k]])
    grads = net.get_gradients()
    for k in grads_ref:
        rep["grad/" + k] = err(grads[k], grads_ref[k])
    return rep
