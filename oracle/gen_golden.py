"""Generates tests/golden/*.npz|json.  Imports the reference's own host-side Python from the original GA3C's ga3c/
directory, which is not part of this repository:

    GA3C_REFERENCE=/path/to/GA3C/ga3c python -m oracle.gen_golden

Pinned against the REAL reference (imported, unmodified):
  returns.json      ProcessAgent._accumulate_rewards  (ProcessAgent.py:70-84) under the default
                    Config and under the three flag variants the function reads
  sampling.npz      ProcessAgent.select_action / np.random.choice (ProcessAgent.py:110-115) driven
                    by a seeded legacy RandomState, with the uniforms it consumed
  convert_data.npz  ProcessAgent.convert_data (ProcessAgent.py:86-100)
Self-pins (oracle_np output frozen so later edits cannot drift silently; the reference cannot run
its TensorFlow graph here, so these are NOT reference outputs -- parity unpinned):
  network_b4.npz    forward / losses / gradient digests / one RMSProp step at B=4, seed 12345
  mlp_b6.npz        the config-4 MLPs (fork NetworkVP S=3 A=1, NetworkVP_discrate S=4 A=2) at B=6: inputs, p / v, the five
                    loss scalars and every gradient, computed by a torch-autograd restatement of the reference graph lines
                    (gen_mlp below, fp64) -- a second, independent statement for oracle_mlp.py and the CUDA path to meet
"""
from __future__ import annotations

import json
import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(os.path.dirname(HERE), "tests", "golden")
REF = os.environ.get("GA3C_REFERENCE", "")


def import_reference_agent():
    """ProcessAgent imports gym/matplotlib/skimage transitively (EnvironmentPend ->
    PyperEnvironment -> pyper_env); stub them so the *unmodified* module imports."""
    if not os.path.isdir(REF):
        raise RuntimeError("GA3C_REFERENCE must name the original GA3C's ga3c/ directory")
    sys.dont_write_bytecode = True
    if REF not in sys.path:
        sys.path.insert(0, REF)
    class _Stub(types.ModuleType):
        """Any attribute resolves to a do-nothing callable / sub-stub (simulator deps only)."""
        __path__ = []

        def __getattr__(self, item):
            if item.startswith("__"):
                raise AttributeError(item)
            return _Stub(self.__name__ + "." + item)

        def __call__(self, *a, **k):
            return None

    for name in ("gym", "gym.wrappers", "matplotlib", "matplotlib.pyplot", "matplotlib.image", "skimage",
                 "skimage.morphology", "skimage.color", "scipy.misc"):
        if name not in sys.modules:
            sys.modules[name] = _Stub(name)
    import ProcessAgent as PA   # noqa
    import Config as CFG        # noqa
    import Experience as EXP    # noqa
    return PA.ProcessAgent, CFG.Config, EXP.Experience


def gen_returns(ProcessAgent, Config, Experience):
    rng = np.random.default_rng(7)
    cases = []
    variants = [
        dict(DISCOUNTING=True, USE_INTERMEDIATE_REWARD=False, REWARD_CLIPPING=True),   # default
        dict(DISCOUNTING=True, USE_INTERMEDIATE_REWARD=True, REWARD_CLIPPING=True),
        dict(DISCOUNTING=False, USE_INTERMEDIATE_REWARD=False, REWARD_CLIPPING=True),
        dict(DISCOUNTING=True, USE_INTERMEDIATE_REWARD=False, REWARD_CLIPPING=False),
    ]
    saved = {k: getattr(Config, k) for k in variants[0]}
    try:
        for var in variants:
            for k, v in var.items():
                setattr(Config, k, v)
            for n in (1, 2, 3, 6, 17, 1001):
                for gamma in (0.99, 0.5):
                    rewards = [float(r) for r in rng.uniform(-3, 3, size=n)]
                    exps = [Experience(None, 0, None, r, None, False) for r in rewards]
                    terminal = rewards[-1]                       # ProcessAgent.py:148
                    out = ProcessAgent._accumulate_rewards(exps, gamma, terminal)
                    cases.append(dict(flags=var, n=n, gamma=gamma, rewards=rewards, terminal=terminal,
                                      out=[float(e.reward).hex() for e in out]))
    finally:
        for k, v in saved.items():
            setattr(Config, k, v)
    with open(os.path.join(GOLD, "returns.json"), "w") as f:
        json.dump(cases, f)
    print("returns.json", len(cases), "cases")


def gen_sampling(ProcessAgent, Config):
    assert not Config.PLAY_MODE
    rng = np.random.default_rng(11)
    n, a_n = 512, 6
    z = rng.normal(0, 2, size=(n, a_n)).astype(np.float32)
    e = np.exp(z - z.max(axis=1, keepdims=True))
    p = (e / e.sum(axis=1, keepdims=True)).astype(np.float32)
    actions = np.arange(a_n)
    np.random.seed(4242)
    chosen = np.array([ProcessAgent.select_action(actions, p[i]) for i in range(n)], dtype=np.int32)
    np.random.seed(4242)
    u = np.array([np.random.random_sample() for _ in range(n)], dtype=np.float64)
    np.savez_compressed(os.path.join(GOLD, "sampling.npz"), p=p, u=u, chosen=chosen)
    print("sampling.npz", n)


def gen_convert(ProcessAgent, Experience):
    rng = np.random.default_rng(13)
    n, s, a_n = 9, 12, 6

    class FakeSelf:       # convert_data only touches self.num_actions
        num_actions = a_n
    exps = []
    for _ in range(n):
        exps.append(Experience(rng.normal(size=s).astype(np.float32), int(rng.integers(0, a_n)),
                               None, float(rng.uniform(-1, 1)), rng.normal(size=s).astype(np.float32),
                               bool(rng.integers(0, 2))))
    x_, r_, a_, x2_, done_ = ProcessAgent.convert_data(FakeSelf(), exps)
    np.savez_compressed(os.path.join(GOLD, "convert_data.npz"),
                        states=np.array([e.state for e in exps]), actions=np.array([e.action for e in exps]),
                        rewards=np.array([e.reward for e in exps]), next_states=np.array([e.next_state for e in exps]),
                        dones=np.array([e.done for e in exps]), x_=x_, r_=r_, a_=a_, x2_=x2_, done_=done_)
    print("convert_data.npz", x_.dtype, r_.dtype, a_.dtype, done_.dtype)


def digest(g):
    g = np.asarray(g, dtype=np.float64).ravel()
    idx = np.linspace(0, g.size - 1, num=min(g.size, 64)).astype(np.int64)
    return dict(sum=float(g.sum()), l2=float(np.sqrt((g * g).sum())), amax=float(np.abs(g).max()),
                idx=idx.tolist(), val=g[idx].tolist())


def gen_network():
    from . import oracle_np as onp
    rng = np.random.default_rng(12345)                      # Config.RANDOM_SEED, Config.py:187
    params = onp.init_params(rng, 6)
    x = onp.synth_frames(rng, 4)
    y_r, a = onp.synth_targets(rng, 4)
    out = {}
    for tag, kw in (("f64", dict(dtype=np.float64)), ("bf16", dict(dtype=np.float64, quant="bf16"))):
        ms, mom = onp.rmsprop_init(params)
        losses, grads, p2, ms2, _ = onp.train_step(params, ms, mom, x, y_r, a, lr=3e-4, **kw)
        p, v = onp.forward(params, x, **kw)
        out[f"{tag}_p"], out[f"{tag}_v"] = p, v
        out[f"{tag}_losses"] = np.array([losses[k] for k in ("cost_p_1", "cost_p_2", "cost_p", "cost_v", "cost_all")])
        out[f"{tag}_digests"] = np.array(json.dumps({k: digest(g) for k, g in grads.items()}))
        out[f"{tag}_post_digests"] = np.array(json.dumps({k: digest(g) for k, g in p2.items()}))
        for k in ("conv11/b:0", "conv12/b:0", "dense1/b:0", "logits_p/w:0", "logits_v/w:0", "conv11/w:0"):
            out[f"{tag}_grad_{k}"] = grads[k]
    np.savez_compressed(os.path.join(GOLD, "network_b4.npz"), **out)
    print("network_b4.npz")


def gen_mlp():
    """torch restatement of NetworkVP.py:79-105 (+ :175-210) and NetworkVP_discrate.py:52-85, autograd for the backward."""
    import torch
    from . import oracle_mlp as om
    out = {}
    for kind, s, a in (("fork_vp", 3, 1), ("discrate", 4, 2)):
        rng = np.random.default_rng(2024)
        params = om.init_params(rng, kind, s, a)
        b = 6
        x = rng.uniform(-1, 1, size=(b, s)).astype(np.float32)
        y_r = rng.uniform(-1, 1, size=b).astype(np.float32)
        act = (rng.uniform(-1, 1, size=(b, a)).astype(np.float32) if kind == "fork_vp"
               else np.eye(a, dtype=np.float32)[rng.integers(0, a, size=b)])
        tp = {k: torch.tensor(v.astype(np.float64), requires_grad=True) for k, v in params.items()}
        tx, tyr, ta = (torch.tensor(np.asarray(t, dtype=np.float64)) for t in (x, y_r, act))
        beta, eps = 0.01, 1e-6
        def dense(h, name, func):
            z = h @ tp[name + "/w:0"] + tp[name + "/b:0"]
            return func(z) if func is not None else z
        if kind == "fork_vp":
            h = dense(tx, "dense11_p", None); h = dense(h, "dense12_p", None); h = dense(h, "dense13_p", None)
            h = dense(h, "dense14_p", torch.sigmoid); h = dense(h, "dense1", torch.sigmoid)
            v = dense(h, "logits_v", None)[:, 0]
            ox = dense(h, "logits_p/out_x", torch.sigmoid) - 0.5
            oy = dense(h, "logits_p/out_y", torch.sigmoid) - 0.5
            p = torch.atan2(oy, ox) / np.pi
            c1 = ((p * ta).sum(1) * (tyr - v.detach())).sum()
            c2 = (-beta * (p * p).sum(1)).sum()
        else:
            h = dense(tx, "dense1_4_p", torch.sigmoid)          # every DENSE_LAYERS entry reads x; the last one is live
            v = dense(h, "logits_v", None)[:, 0]
            p = torch.softmax(dense(h, "logits_p", None), dim=1)
            c1 = (torch.log(torch.clamp((p * ta).sum(1), min=eps)) * (tyr - v.detach())).sum()
            c2 = (-beta * (torch.log(torch.clamp(p, min=eps)) * p).sum(1)).sum()
        cv = 0.5 * ((tyr - v) ** 2).sum()
        total = -(c1 + c2) + cv
        total.backward()
        out[f"{kind}_x"], out[f"{kind}_yr"], out[f"{kind}_a"] = x, y_r, act
        out[f"{kind}_p"], out[f"{kind}_v"] = p.detach().numpy(), v.detach().numpy()
        out[f"{kind}_losses"] = np.array([float(c1), float(c2), float(-(c1 + c2)), float(cv), float(total)])
        for k, t in tp.items():                 # weights are om.init_params(default_rng(2024), kind, s, a): not stored
            if t.grad is not None:
                out[f"{kind}_grad_{k}"] = t.grad.numpy().astype(np.float32)
    np.savez_compressed(os.path.join(GOLD, "mlp_b6.npz"), **out)
    print("mlp_b6.npz")


def main():
    os.makedirs(GOLD, exist_ok=True)
    if "--mlp-only" in sys.argv:
        return gen_mlp()
    ProcessAgent, Config, Experience = import_reference_agent()
    gen_returns(ProcessAgent, Config, Experience)
    gen_sampling(ProcessAgent, Config)
    gen_convert(ProcessAgent, Experience)
    gen_network()
    gen_mlp()


if __name__ == "__main__":
    main()
