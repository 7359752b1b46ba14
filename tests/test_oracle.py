"""CPU tests pinning the oracle (`-m "not gpu"`).

 * host-side functions: bit-exact against golden vectors produced by the REAL reference code
   (oracle/gen_golden.py), and live against $GA3C_REFERENCE where it is set;
 * network arithmetic (parity unpinned by the reference): finite differences, torch autograd as
   an independent second opinion, and a frozen self-pin.
"""
import json
import os

import numpy as np
import pytest
import torch

from oracle import oracle_np as onp
from oracle.oracle_torch import TorchNetworkVP


# ---------------------------------------------------------------- geometry / rounding
def test_same_padding_geometry():
    assert (onp.H1, onp.P1_LO, onp.P1_HI) == (21, 2, 2)          # SURVEY A.1
    assert (onp.H2, onp.P2_LO, onp.P2_HI) == (11, 1, 2)          # asymmetric
    assert onp.FLAT == 3872
    n = sum(int(np.prod(s)) for s in onp.param_shapes(6).values())
    assert n == 1005623


def test_bf16_round_matches_torch():
    rng = np.random.default_rng(0)
    x = np.concatenate([rng.normal(size=4096), rng.normal(size=64) * 1e-30, [0.0, -0.0, 1.0, 65280.0]]).astype(np.float32)
    ref = torch.from_numpy(x).to(torch.bfloat16).to(torch.float32).numpy()
    assert np.array_equal(onp.bf16_round(x), ref)


def test_synthetic_frames_are_exact_in_bf16():
    x = onp.synth_frames(np.random.default_rng(1), 2)
    assert np.array_equal(onp.bf16_round(x), x)                     # k/128-1 needs 8 significand bits
    assert x.min() >= -1.0 and x.max() <= 127 / 128


# ---------------------------------------------------------------- golden: real reference outputs
def test_returns_golden_bit_exact(golden_dir):
    cases = json.load(open(os.path.join(golden_dir, "returns.json")))
    assert len(cases) == 48
    for c in cases:
        f = c["flags"]
        out = onp.accumulate_rewards(c["rewards"], c["gamma"], c["terminal"], discounting=f["DISCOUNTING"],
                                     use_intermediate_reward=f["USE_INTERMEDIATE_REWARD"],
                                     reward_clipping=f["REWARD_CLIPPING"])
        assert [float(r).hex() for r in out] == c["out"]


def test_returns_default_closed_form(golden_dir):
    """SURVEY A.7: R_t = gamma^(n-1-t) * r_last by repeated multiplication."""
    out = onp.accumulate_rewards([0.3, -2.0, 0.7, 0.25], 0.99, 0.25)
    assert out[3] == 0.25 and out[2] == 0.99 * 0.25 and out[1] == 0.99 * (0.99 * 0.25)
    assert onp.accumulate_rewards([], 0.99, 1.0) == [] and onp.accumulate_rewards([5.0], 0.99, 5.0) == [5.0]


def test_sampling_golden_bit_exact(golden_dir):
    g = np.load(os.path.join(golden_dir, "sampling.npz"))
    got = onp.select_actions(g["p"], g["u"])
    assert np.array_equal(got, g["chosen"])


def test_convert_data_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "convert_data.npz"))
    assert g["r_"].dtype == np.float64 and g["a_"].dtype == np.float32    # SURVEY Appendix B
    assert np.array_equal(np.eye(6)[g["actions"]].astype(np.float32), g["a_"])
    assert np.array_equal(g["states"], g["x_"]) and np.array_equal(g["rewards"], g["r_"])


# ---------------------------------------------------------------- live against the reference
@pytest.mark.reference
def test_returns_live_against_reference():
    from oracle.gen_golden import import_reference_agent
    ProcessAgent, Config, Experience = import_reference_agent()
    rng = np.random.default_rng(99)
    for n in (1, 2, 5, 64, 300):
        rewards = [float(r) for r in rng.uniform(-2, 2, size=n)]
        exps = [Experience(None, 0, None, r, None, False) for r in rewards]
        ref = [e.reward for e in ProcessAgent._accumulate_rewards(exps, Config.DISCOUNT, rewards[-1])]
        assert ref == onp.accumulate_rewards(rewards, Config.DISCOUNT, rewards[-1])


# ---------------------------------------------------------------- network arithmetic
@pytest.fixture(scope="module")
def small():
    rng = np.random.default_rng(12345)
    params = onp.init_params(rng, 6)
    x = onp.synth_frames(rng, 4)
    y_r, a = onp.synth_targets(rng, 4)
    return params, x, y_r, a


def test_backward_matches_torch_autograd_fp64(small):
    params, x, y_r, a = small
    losses, grads = onp.loss_and_grads(params, x, y_r, a, beta=0.01)
    tl, tg = TorchNetworkVP(params, dtype=torch.float64).grads(x, y_r, a, 0.01)
    for k in losses:
        assert abs(losses[k] - tl[k]) <= 1e-12 * max(1.0, abs(tl[k]))
    for k in grads:
        assert np.abs(grads[k] - tg[k]).max() <= 1e-12, k


def test_backward_matches_torch_with_min_policy_and_floor(small):
    """MIN_POLICY mixing and an epsilon floor large enough to be active (mask branches of A.4)."""
    params, x, y_r, a = small
    kw = dict(beta=0.05, log_eps=0.12, min_policy=0.02)
    losses, grads = onp.loss_and_grads(params, x, y_r, a, **kw)
    tn = TorchNetworkVP(params, dtype=torch.float64, log_eps=0.12, min_policy=0.02)
    tl, tg = tn.grads(x, y_r, a, 0.05)
    assert abs(losses["cost_all"] - tl["cost_all"]) < 1e-12
    for k in grads:
        assert np.abs(grads[k] - tg[k]).max() <= 1e-12, k


def test_backward_finite_differences(small):
    params, x, y_r, a = small
    p64 = {k: v.astype(np.float64) for k, v in params.items()}
    _, grads = onp.loss_and_grads(p64, x, y_r, a)
    _, v0 = onp.forward(p64, x)

    def f(pm):
        p, v = onp.forward(pm, x)
        return onp.losses_from_heads(p, v, y_r.astype(np.float64), a.astype(np.float64), 0.01, 1e-6, v_stop=v0)["cost_all"]

    rng = np.random.default_rng(5)
    for k in p64:
        for _ in range(3):
            idx = tuple(int(rng.integers(0, s)) for s in p64[k].shape)
            if grads[k][idx] == 0.0:
                continue
            h = 1e-5
            pp = {n: v.copy() for n, v in p64.items()}
            pm = {n: v.copy() for n, v in p64.items()}
            pp[k][idx] += h
            pm[k][idx] -= h
            fd = (f(pp) - f(pm)) / (2 * h)
            assert abs(fd - grads[k][idx]) <= 1e-6 * max(1.0, abs(fd)), (k, idx, fd, grads[k][idx])


def test_log_softmax_branch_finite_differences_and_torch(small):
    """Config.USE_LOG_SOFTMAX (NetworkVP_discrate.py:64-71): analytic backward against finite differences (advantage frozen,
    tf.stop_gradient) and against torch autograd on log_softmax / softmax of the oracle's own logits."""
    params, x, y_r, a = small
    p64 = {k: v.astype(np.float64) for k, v in params.items()}
    a = a.astype(np.float64) * 0.7 + 0.05                     # not one-hot: exercises the sum(a) term
    losses, grads, f = onp.loss_and_grads(p64, x, y_r, a, beta=0.03, use_log_softmax=True, keep=True)
    p, _ = onp.forward(p64, x, use_log_softmax=True)
    assert np.allclose(p.sum(axis=1), 1.0) and np.array_equal(p, f["s"])
    v0 = f["v"]

    def cost(pm):
        g = onp.forward(pm, x, keep=True, use_log_softmax=True)
        return onp.losses_from_log_softmax(g["lsm"], g["s"], g["v"], y_r.astype(np.float64), a, 0.03, v_stop=v0)["cost_all"]

    rng = np.random.default_rng(9)
    for k in p64:
        for _ in range(3):
            idx = tuple(int(rng.integers(0, s)) for s in p64[k].shape)
            if grads[k][idx] == 0.0:
                continue
            h = 1e-7                                            # small: a ReLU kink inside (-h, h) spoils the difference
            pp = {n: v.copy() for n, v in p64.items()}; pp[k][idx] += h
            pm = {n: v.copy() for n, v in p64.items()}; pm[k][idx] -= h
            fd = (cost(pp) - cost(pm)) / (2 * h)
            assert abs(fd - grads[k][idx]) <= 1e-6 * max(1.0, abs(fd)), (k, idx, fd, grads[k][idx])
    z = torch.tensor(f["z"], requires_grad=True)
    v = torch.tensor(f["v"], requires_grad=True)
    yr, at = torch.tensor(y_r.astype(np.float64)), torch.tensor(a)
    lsm, sm = torch.log_softmax(z, dim=1), torch.softmax(z, dim=1)
    c1 = ((lsm * at).sum(1) * (yr - v.detach())).sum()
    c2 = (-0.03 * (lsm * sm).sum(1)).sum()
    total = -(c1 + c2) + 0.5 * ((yr - v) ** 2).sum()
    total.backward()
    assert abs(float(total) - losses["cost_all"]) <= 1e-10 * max(1.0, abs(losses["cost_all"]))
    assert np.abs(z.grad.numpy() - f["dz"]).max() <= 1e-12 and np.abs(v.grad.numpy() - f["dv"]).max() <= 1e-12


def test_dual_rmsprop_gradients_split_cost_p_and_cost_v(small):
    """Config.DUAL_RMSPROP: the two gradients add up to the (pinned) gradient of cost_all, cost_v's gradient matches finite
    differences of cost_v alone, and each cost leaves the other head's variables without a gradient."""
    params, x, y_r, a = small
    p64 = {k: v.astype(np.float64) for k, v in params.items()}
    _, g_all = onp.loss_and_grads(p64, x, y_r, a)
    _, g_p = onp.loss_and_grads(p64, x, y_r, a, part="p")
    _, g_v = onp.loss_and_grads(p64, x, y_r, a, part="v")
    assert set(g_all) - set(g_p) == {"logits_v/w:0", "logits_v/b:0"} and set(g_all) - set(g_v) == {"logits_p/w:0", "logits_p/b:0"}
    for k in g_all:
        tot = g_p.get(k, 0.0) + g_v.get(k, 0.0)
        assert np.abs(tot - g_all[k]).max() <= 1e-12 * max(1.0, np.abs(g_all[k]).max()), k

    def cost_v(pm):
        _, v = onp.forward(pm, x)
        return 0.5 * ((y_r.astype(np.float64) - v) ** 2).sum()

    rng = np.random.default_rng(3)
    for k in g_v:
        for _ in range(3):
            idx = tuple(int(rng.integers(0, s)) for s in p64[k].shape)
            if g_v[k][idx] == 0.0:
                continue
            h = 1e-7
            pp = {n: v.copy() for n, v in p64.items()}; pp[k][idx] += h
            pm = {n: v.copy() for n, v in p64.items()}; pm[k][idx] -= h
            fd = (cost_v(pp) - cost_v(pm)) / (2 * h)
            assert abs(fd - g_v[k][idx]) <= 1e-6 * max(1.0, abs(fd)), (k, idx, fd, g_v[k][idx])
    # one dual step: both steps from the pre-call weights, untouched variables keep their slots
    ms, mom = onp.rmsprop_init(p64)
    _, gp, gv, new_p, (ms_p, _), (ms_v, _) = onp.train_step_dual(p64, (ms, mom), (ms, mom), x, y_r, a, lr=1e-2)
    k = "conv11/b:0"
    exp = p64[k] - 1e-2 * gp[k] / np.sqrt(0.99 + 0.01 * gp[k] ** 2 + 0.1) - 1e-2 * gv[k] / np.sqrt(0.99 + 0.01 * gv[k] ** 2 + 0.1)
    assert np.allclose(new_p[k], exp, rtol=0, atol=1e-14)
    assert np.array_equal(ms_p["logits_v/w:0"], ms["logits_v/w:0"]) and np.array_equal(ms_v["logits_p/w:0"], ms["logits_p/w:0"])


def test_clip_by_average_norm_known_answers():
    """tf.clip_by_average_norm: t * clip / max(||t|| / n, clip)  [TF-SEMANTICS]."""
    g = np.array([[3.0, 4.0]], dtype=np.float32)                       # ||g|| = 5, n = 2 -> average norm 2.5
    assert np.allclose(onp.clip_by_average_norm(g, 1.0), g / 2.5)
    assert np.array_equal(onp.clip_by_average_norm(g, 2.5), g)         # at the threshold: unchanged
    assert np.array_equal(onp.clip_by_average_norm(g, 40.0), g)        # Config.GRAD_CLIP_NORM = 40: never active in practice
    assert onp.clip_by_average_norm(g, 1.0).dtype == np.float32
    t = torch.tensor(g)
    ref = t * 1.0 / torch.maximum(torch.linalg.vector_norm(t) / t.numel(), torch.tensor(1.0))
    assert np.allclose(onp.clip_by_average_norm(g, 1.0), ref.numpy())


def test_clip_by_norm_known_answers_and_dual_clip_step(small):
    """tf.clip_by_norm: t * clip / max(||t||, clip) [TF-SEMANTICS]; DUAL_RMSPROP + USE_GRAD_CLIP clips every variable's gradient
    of each optimizer before its own RMSProp step (NetworkVP_discrate.py:107-117)."""
    g = np.array([[3.0, 4.0]])
    assert np.allclose(onp.clip_by_norm(g, 1.0), g / 5.0) and np.array_equal(onp.clip_by_norm(g, 5.0), g)
    t = torch.tensor(g)
    assert np.allclose(onp.clip_by_norm(g, 2.0), (t * 2.0 / torch.clamp(torch.linalg.vector_norm(t), min=2.0)).numpy())
    params, x, y_r, a = small
    p64 = {k: v.astype(np.float64) for k, v in params.items()}
    ms, mom = onp.rmsprop_init(p64)
    clip = 1e-2
    _, gp, gv, new_p, _, _ = onp.train_step_dual(p64, (ms, mom), (ms, mom), x, y_r, a, lr=1e-2, grad_clip=clip)
    k = "dense1/b:0"
    cp, cv = onp.clip_by_norm(gp[k], clip), onp.clip_by_norm(gv[k], clip)
    assert np.sqrt((gp[k] ** 2).sum()) > clip                           # the clip is active on this variable
    exp = p64[k] - 1e-2 * cp / np.sqrt(0.99 + 0.01 * cp ** 2 + 0.1) - 1e-2 * cv / np.sqrt(0.99 + 0.01 * cv ** 2 + 0.1)
    assert np.allclose(new_p[k], exp, rtol=0, atol=1e-14)


def test_rmsprop_tf_semantics():
    """eps inside the sqrt, ms initialised to 1.0 (SURVEY A.5)."""
    w = {"w": np.array([1.0, -2.0], dtype=np.float32)}
    g = {"w": np.array([0.5, 4.0], dtype=np.float32)}
    ms, mom = onp.rmsprop_init(w)
    w2, ms2, _ = onp.rmsprop_update(w, g, ms, mom, lr=0.1, dtype=np.float64)
    exp_ms = 0.99 * 1.0 + 0.01 * np.array([0.25, 16.0])
    assert np.allclose(ms2["w"], exp_ms, rtol=0, atol=1e-7)
    assert np.allclose(w2["w"], np.array([1.0, -2.0]) - 0.1 * np.array([0.5, 4.0]) / np.sqrt(exp_ms + 0.1), atol=1e-7)


def test_network_self_pin(small, golden_dir):
    params, x, y_r, a = small
    g = np.load(os.path.join(golden_dir, "network_b4.npz"))
    for tag, kw in (("f64", {}), ("bf16", dict(quant="bf16"))):
        p, v = onp.forward(params, x, **kw)
        assert np.allclose(p, g[f"{tag}_p"], rtol=0, atol=1e-12)
        assert np.allclose(v, g[f"{tag}_v"], rtol=0, atol=1e-12)
        losses, grads = onp.loss_and_grads(params, x, y_r, a, **kw)
        got = np.array([losses[k] for k in ("cost_p_1", "cost_p_2", "cost_p", "cost_v", "cost_all")])
        assert np.allclose(got, g[f"{tag}_losses"], rtol=1e-12)
        dig = json.loads(str(g[f"{tag}_digests"]))
        for k, d in dig.items():
            flat = grads[k].ravel()
            assert np.allclose(flat[d["idx"]], d["val"], rtol=1e-9, atol=1e-14), k
            assert abs(flat.sum() - d["sum"]) <= 1e-9 * max(1.0, abs(d["sum"]))


def test_bf16_mode_is_close_to_fp64(small):
    params, x, _, _ = small
    p, v = onp.forward(params, x)
    pq, vq = onp.forward(params, x, quant="bf16")
    assert np.abs(p - pq).max() < 5e-3 and np.abs(v - vq).max() < 5e-3
    assert np.abs(p.sum(axis=1) - 1).max() < 1e-12


def test_tf_reference_pin(golden_dir):
    """Opt-in pin against the REAL reference: tests/golden/tf_reference_b4.npz is written by tools/dump_tf_reference.py on a box
    that has TensorFlow (this build container has none, so the file does not exist yet and the network arithmetic stays
    'parity unpinned').  When present: the oracle in fp32 must reproduce TensorFlow's fp32 graph -- predictions, the five
    loss scalars, all ten gradients, and weights / RMSProp slots after one train step -- which settles every [TF-SEMANTICS]
    assumption at once (SAME padding split, tf.maximum sub-gradient, epsilon inside the sqrt, ms initialised to 1)."""
    import os
    path = os.path.join(golden_dir, "tf_reference_b4.npz")
    if not os.path.exists(path):
        pytest.skip("no TensorFlow dump committed (tools/dump_tf_reference.py needs a TensorFlow box)")
    g = np.load(path)
    from _parity import make_case
    params, x, y_r, a = make_case(int(g["batch"]))
    lr, beta = float(g["lr"]), float(g["beta"])
    p, v = onp.forward(params, x, dtype=np.float32)
    assert np.abs(p - g["p"]).max() <= 1e-5 and np.abs(v - g["v"]).max() <= 1e-4 * max(1.0, np.abs(g["v"]).max())
    ms, mom = onp.rmsprop_init(params)
    losses, grads, p2, ms2, mom2 = onp.train_step(params, ms, mom, x, y_r, a, lr=lr, beta=beta, dtype=np.float32)
    got = np.array([losses[k] for k in ("cost_p_1", "cost_p_2", "cost_p", "cost_v", "cost_all")])
    assert np.allclose(got, g["losses"], rtol=1e-4, atol=1e-5)
    for k in onp.PARAM_NAMES:
        ref = g["grad_" + k]
        assert np.abs(grads[k] - ref).max() <= 1e-4 * max(np.abs(ref).max(), 1e-30), k
        assert np.abs(p2[k] - g["after_" + k]).max() <= 1e-6, k
        assert np.allclose(ms2[k], g["after_" + k.replace(":0", "/RMSProp:0")], rtol=1e-4), k
    assert int(g["after_step:0"]) == 1
