"""Shared helpers of the GPU parity tests: run the CUDA path and the oracle on the same seeded
inputs and report per-tensor error figures.  The oracle is the checker, never the thing measured.

Tolerances of the conv network (SURVEY A.8, calibrated on B200 and frozen here).  The CUDA path rounds
operands to bf16 at fixed points (x, conv weights, n1, n2, w1, dd1, dn2, dn1) and accumulates in fp32;
the oracle is run in its `quant='bf16'` mode, which rounds at the same points and accumulates in fp64.
Residual differences are fp32-vs-fp64 accumulation order, which now and then flips a bf16 rounding
(1 ulp = 2^-8 relative) of a stored activation:
    p        |d| <= 2e-5          v        |d| <= 2e-4
    stored bf16 activations      |d| <= 2^-7 * max|ref|  and  <= 1% of elements off by > 1e-5 * max|ref|
    loss sums                    rel <= 1e-4
    gradients                    |d| <= 2e-3 * max|ref| per tensor
    weights after RMSProp        |d| <= 2e-6   (lr 3e-4 scales the gradient error)
Against the un-quantised fp64 oracle (the irreducible bf16 gap): |dp| <= 1e-2, |dv| <= 2e-2.
"""
from __future__ import annotations

import numpy as np
import pytest

from oracle import oracle_mlp as om
from oracle import oracle_np as onp

TOL_P, TOL_V = 2e-5, 2e-4
TOL_ACT_REL = 2.0 ** -7
TOL_LOSS_REL = 1e-4
TOL_GRAD_REL = 2e-3
TOL_W_ABS = 2e-6


@pytest.fixture(scope="module")
def ga3c():
    """The package, for a test module that imports this fixture; fails (never skips) without a CUDA device."""
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; there is no CPU fallback")
    import ga3c_b200
    return ga3c_b200


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


def layer_report(net, params, x, y_r, a, *, geom=None, beta=0.01, log_eps=1e-6, min_policy=0.0, use_log_softmax=False):
    """Runs predict + forward_backward on the conv `net` (weights := params) and compares every stored
    activation, every gradient and the loss sums with the bf16-rounding-point oracle (fp64 accumulate) at
    input geometry `geom` (None: 84x84x4).  Returns {name: (abs_err, rel_err)}."""
    g = onp.DEFAULT_GEOMETRY if geom is None else geom
    net.set_variables(params)
    net.beta = beta
    rep = {}
    p, v = net.predict_p_and_v(x)
    losses_ref, grads_ref, f = onp.loss_and_grads(params, x, y_r, a, geom=g, beta=beta, log_eps=log_eps,
                                                  min_policy=min_policy, quant="bf16", keep=True,
                                                  use_log_softmax=use_log_softmax)
    rep["p"] = err(p, f["p"])
    rep["v"] = err(v, f["v"])
    net.keep_dn1(True)          # dn1 is consumed on chip by the fused conv backward; ask for a copy
    losses = net.losses(x, y_r, a)
    net.keep_dn1(False)
    b = x.shape[0]
    ws = [net.workspace(i) for i in range(6)]
    rep["n1"] = err(ws[0], f["n1"].reshape(b, -1))
    rep["n2"] = err(ws[1], f["n2"].reshape(b, -1))
    rep["d1"] = err(ws[2], f["d1"])
    rep["dd1"] = err(ws[3], f["dd1"])
    rep["dn2"] = err(ws[4], f["dn2"])
    rep["dn1"] = err(ws[5], f["dn1"])
    # Layer-local view of the two masked data gradients: the same oracle arithmetic applied to the CUDA path's OWN stored inputs
    # (dd1 / dn2 and the activation masks).  A stored activation that sits within an fp32-vs-fp64 accumulation difference of
    # the ReLU boundary flips its mask bit; the global comparison above then shows that element's whole gradient (and what
    # it spreads to upstream) as an error although every kernel did its arithmetic right.  At full-size batches (millions of
    # activations) a handful of such flips is certain; the local view is immune, and `outliers` says how few elements differ.
    n1_mask = ws[0].reshape(b, -1) > 0
    n2_mask = ws[1].reshape(b, -1) > 0
    dn2_cuda = ws[4].astype(np.float64).reshape(-1, onp.C2_OUT)
    dd1_cuda = ws[3].astype(np.float64).reshape(b, -1)
    dn2_local = onp.bf16_round((dd1_cuda @ f["w1"].T) * n2_mask)
    n_out, lo, hi = zip(onp.same_pad(g.h1, onp.C2_K, onp.C2_S), onp.same_pad(g.w1, onp.C2_K, onp.C2_S))
    dn1_local = onp._col2im(dn2_cuda @ f["w12"].T, b, (g.h1, g.w1), onp.C2_K, onp.C2_S, lo, hi, n_out, onp.C1_OUT)
    dn1_local = onp.bf16_round(dn1_local.reshape(b, -1) * n1_mask)
    rep["dn2_local"] = err(ws[4], dn2_local)
    rep["dn1_local"] = err(ws[5], dn1_local)
    for k, got in (("dn1", ws[5]), ("dn2", ws[4])):
        ref = np.asarray(f[k], dtype=np.float64).ravel()
        rep[k + "_outliers"] = (float((np.abs(got.ravel() - ref) > 2.0 ** -7 * np.abs(ref).max()).mean()), 0.0)
    for k in ("cost_p_1", "cost_p_2", "cost_v", "cost_all"):
        rep["loss/" + k] = err([losses[k]], [losses_ref[k]])
    grads = net.get_gradients()
    for k in grads_ref:
        rep["grad/" + k] = err(grads[k], grads_ref[k])
    return rep


def check_report(rep):
    """layer_report's figures against the tolerances above."""
    assert rep["p"][0] <= TOL_P and rep["v"][0] <= TOL_V, rep
    for k in ("n1", "n2", "dd1"):
        assert rep[k][1] <= TOL_ACT_REL, (k, rep[k])
    for k in ("dn2", "dn1"):
        # masked data gradients: exact against the oracle fed the same stored inputs; against the end-to-end oracle either
        # within tolerance everywhere, or off only at the rare elements behind a ReLU-boundary flip (layer_report)
        assert rep[k + "_local"][1] <= TOL_ACT_REL, (k, rep[k + "_local"])
        assert rep[k][1] <= TOL_ACT_REL or rep[k + "_outliers"][0] <= 1e-4, (k, rep[k], rep[k + "_outliers"])
    assert rep["d1"][1] <= 1e-3, rep["d1"]
    for k, (d, r) in rep.items():
        if k.startswith("loss/"):
            assert r <= TOL_LOSS_REL or d <= 1e-5, (k, d, r)
        if k.startswith("grad/"):
            assert r <= TOL_GRAD_REL, (k, d, r)
