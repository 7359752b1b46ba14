"""numpy restatement of the GA3C conv NetworkVP hot path.  TEST INFRASTRUCTURE ONLY.

PARITY UNPINNED for the network arithmetic: the reference delegates it to an
un-vendored, un-pinned TensorFlow 1.x (README.md:8).  This file restates the
graph from the reference's own call sites (all paths below are into
/root/reference/ga3c):

  conv layer       NetworkVP.py:212-228   (HWIO weights, SAME padding, bias, ReLU)
  trunk topology   NetworkDNav.py:81-90   (conv11 8x8/16/s4 -> conv12 4x4/32/s2 -> flat -> dense1 256)
  dense layer      NetworkDNav.py:256-269 (x @ w + b, ReLU)
  heads + loss     NetworkVP_discrate.py:60-85, :100
  optimizer        NetworkVP_discrate.py:101-105 (tf.train.RMSPropOptimizer, non-centred)
  returns          ProcessAgent.py:70-84
  sampling         ProcessAgent.py:110-115  (np.random.choice)

Three arithmetic modes:
  dtype=np.float64, quant=None   -- the mathematical oracle (finite-difference checked)
  dtype=np.float32, quant=None   -- what fp32 TF would compute, up to summation order
  quant='bf16'                   -- operands rounded to bfloat16 at exactly the points where
                                    the CUDA path rounds them (see DESIGN.md "Rounding points");
                                    accumulation stays in `dtype`.

The input geometry (Config.IMAGE_HEIGHT, IMAGE_WIDTH, STACKED_FRAMES) is the keyword `geom=`, a Geometry; None means
the reference's 84x84x4, whose sizes are also the module constants below.
"""
from __future__ import annotations

import numpy as np

# --------------------------------------------------------------------------------------
# geometry
# --------------------------------------------------------------------------------------
H = W = 84
C = 4
STATE_DIM = H * W * C          # 28224, Config.py:90-92
C1_K, C1_S, C1_OUT = 8, 4, 16  # NetworkDNav.py:81
C2_K, C2_S, C2_OUT = 4, 2, 32  # NetworkDNav.py:82
FC = 256                       # NetworkDNav.py:90

# TF variable names in creation order (what get_variables_names() returns, NetworkVP.py:284-285)
PARAM_NAMES = (
    "conv11/w:0", "conv11/b:0", "conv12/w:0", "conv12/b:0", "dense1/w:0", "dense1/b:0",
    "logits_v/w:0", "logits_v/b:0", "logits_p/w:0", "logits_p/b:0",
)


def same_pad(n_in: int, k: int, s: int):
    """TF 'SAME' padding [TF-SEMANTICS]: out = ceil(in/s), pad split low-side-smaller."""
    out = -(-n_in // s)
    total = max((out - 1) * s + k - n_in, 0)
    before = total // 2
    return out, before, total - before


H1, P1_LO, P1_HI = same_pad(H, C1_K, C1_S)    # 21, 2, 2
H2, P2_LO, P2_HI = same_pad(H1, C2_K, C2_S)   # 11, 1, 2
FLAT = H2 * H2 * C2_OUT                       # 3872


class Geometry:
    """Derived sizes of an h x w x c input under TF SAME padding (SURVEY A.1): conv11's output h1 x w1 with top / left pads
    pt1 / pl1, conv12's h2 x w2 with pt2 / pl2, and dense1's fan-in flat = h2 * w2 * 32."""

    def __init__(self, h: int, w: int, c: int):
        self.h, self.w, self.c = h, w, c
        self.h1, self.pt1, _ = same_pad(h, C1_K, C1_S)
        self.w1, self.pl1, _ = same_pad(w, C1_K, C1_S)
        self.h2, self.pt2, _ = same_pad(self.h1, C2_K, C2_S)
        self.w2, self.pl2, _ = same_pad(self.w1, C2_K, C2_S)
        self.state_dim = h * w * c
        self.flat = self.h2 * self.w2 * C2_OUT

    def __repr__(self):
        return f"{self.h}x{self.w}x{self.c}"


DEFAULT_GEOMETRY = Geometry(H, W, C)


def _geom(geom):
    return DEFAULT_GEOMETRY if geom is None else geom


def param_shapes(num_actions: int, *, geom=None):
    g = _geom(geom)
    return {
        "conv11/w:0": (C1_K, C1_K, g.c, C1_OUT), "conv11/b:0": (C1_OUT,),
        "conv12/w:0": (C2_K, C2_K, C1_OUT, C2_OUT), "conv12/b:0": (C2_OUT,),
        "dense1/w:0": (g.flat, FC), "dense1/b:0": (FC,),
        "logits_v/w:0": (FC, 1), "logits_v/b:0": (1,),
        "logits_p/w:0": (FC, num_actions), "logits_p/b:0": (num_actions,),
    }


def init_params(rng: np.random.Generator, num_actions: int = 6, *, geom=None):
    """U(-d, d) with d = 1/sqrt(fan_in): NetworkVP.py:214-217 (conv), NetworkDNav.py:258-261 (dense)."""
    g = _geom(geom)
    fan_in = {"conv11": C1_K * C1_K * g.c, "conv12": C2_K * C2_K * C1_OUT, "dense1": g.flat,
              "logits_v": FC, "logits_p": FC}
    out = {}
    for name, shp in param_shapes(num_actions, geom=g).items():
        d = 1.0 / np.sqrt(fan_in[name.split("/")[0]])
        out[name] = rng.uniform(-d, d, size=shp).astype(np.float32)
    return out


def normalise(k):
    """Environment.py:57-61: uint8 k -> k/128 - 1 (float32)."""
    return (k.astype(np.float32) / np.float32(128.0) - np.float32(1.0)).astype(np.float32)


def synth_frames(rng: np.random.Generator, batch: int, *, geom=None):
    """Frames exactly as Environment.py produces them, drawn as int64."""
    return normalise(rng.integers(0, 256, size=(batch, _geom(geom).state_dim), dtype=np.int64))


def synth_frames_u8(rng: np.random.Generator, batch: int, *, geom=None):
    """The uint8 frames themselves (a different draw from synth_frames'); normalise() gives their float32 form."""
    return rng.integers(0, 256, size=(batch, _geom(geom).state_dim), dtype=np.uint8)


def synth_targets(rng: np.random.Generator, batch: int, num_actions: int = 6):
    y_r = rng.uniform(-1.0, 1.0, size=batch).astype(np.float32)
    idx = rng.integers(0, num_actions, size=batch)
    a = np.eye(num_actions, dtype=np.float32)[idx]   # ProcessAgent.py:98
    return y_r, a


# --------------------------------------------------------------------------------------
# bfloat16 rounding (round-to-nearest-even on the top 16 bits of an IEEE float32)
# --------------------------------------------------------------------------------------
def bf16_round(x):
    x32 = np.ascontiguousarray(x, dtype=np.float32)
    u = x32.view(np.uint32).astype(np.uint64)
    lsb = (u >> 16) & 1
    u = (u + 0x7FFF + lsb) & 0xFFFF0000
    return u.astype(np.uint32).view(np.float32).reshape(x32.shape)


def _q(x, quant, dtype):
    if quant == "bf16":
        return bf16_round(x).astype(dtype)
    return np.asarray(x, dtype=dtype)


# --------------------------------------------------------------------------------------
# conv as im2col (cross-correlation, NHWC x HWIO, SAME) -- NetworkVP.py:224
# --------------------------------------------------------------------------------------
def _im2col(x, k, s):
    """x [B, H, W, C] -> [B*OH*OW, k*k*C] for a k x k / stride s conv with SAME zero padding."""
    b, h, w, c = x.shape
    oh, t, bo = same_pad(h, k, s)
    ow, l, r = same_pad(w, k, s)
    xp = np.zeros((b, h + t + bo, w + l + r, c), dtype=x.dtype)
    xp[:, t:t + h, l:l + w, :] = x
    sb, sh, sw, sc = xp.strides
    cols = np.lib.stride_tricks.as_strided(
        xp, shape=(b, oh, ow, k, k, c), strides=(sb, sh * s, sw * s, sh, sw, sc), writeable=False)
    return cols.reshape(b * oh * ow, k * k * c)     # K order (kh, kw, cin)


def _col2im(dcols, b, h, k, s, lo, hi, n_out, c):
    """The adjoint of _im2col: dcols [B*OH*OW, k*k*c] summed back onto the unpadded [B, H, W, c] input.  The input size h,
    the SAME pads lo / hi and the output size n_out are one int each for a square input, else (vertical, horizontal) pairs."""
    (h, w), (t, l), (bo, r), (oh, ow) = (np.broadcast_to(v, 2) for v in (h, lo, hi, n_out))
    dxp = np.zeros((b, h + t + bo, w + l + r, c), dtype=dcols.dtype)
    d6 = dcols.reshape(b, oh, ow, k, k, c)
    for kh in range(k):
        for kw in range(k):
            dxp[:, kh:kh + s * oh:s, kw:kw + s * ow:s, :] += d6[:, :, :, kh, kw, :]
    return dxp[:, t:t + h, l:l + w, :]


# --------------------------------------------------------------------------------------
# forward
# --------------------------------------------------------------------------------------
def forward(params, x, *, geom=None, dtype=np.float64, quant=None, min_policy=0.0, keep=False, use_log_softmax=False):
    """A2/A3/A4 forward.  x: [B, H*W*C] (flat NHWC).  Returns (p [B,A], v [B]) or a cache dict."""
    g = _geom(geom)
    b = x.shape[0]
    xq = _q(x.reshape(b, g.h, g.w, g.c), quant, dtype)
    w11 = _q(params["conv11/w:0"], quant, dtype).reshape(-1, C1_OUT)
    w12 = _q(params["conv12/w:0"], quant, dtype).reshape(-1, C2_OUT)
    w1 = _q(params["dense1/w:0"], quant, dtype)
    col1 = _im2col(xq, C1_K, C1_S)
    n1 = np.maximum(col1 @ w11 + params["conv11/b:0"].astype(dtype), 0)
    n1 = _q(n1, quant, dtype).reshape(b, g.h1, g.w1, C1_OUT)
    col2 = _im2col(n1, C2_K, C2_S)
    n2 = np.maximum(col2 @ w12 + params["conv12/b:0"].astype(dtype), 0)
    n2 = _q(n2, quant, dtype)
    flat = n2.reshape(b, g.flat)                              # (h, w, c) order, NetworkDNav.py:86-89
    d1 = np.maximum(flat @ w1 + params["dense1/b:0"].astype(dtype), 0)   # stays in `dtype`
    v = (d1 @ params["logits_v/w:0"].astype(dtype) + params["logits_v/b:0"].astype(dtype))[:, 0]
    z = d1 @ params["logits_p/w:0"].astype(dtype) + params["logits_p/b:0"].astype(dtype)
    zs = z - z.max(axis=1, keepdims=True)
    e = np.exp(zs)
    s = e / e.sum(axis=1, keepdims=True)
    a_n = z.shape[1]
    if use_log_softmax:
        p = s                                                              # NetworkVP_discrate.py:65 (no MIN_POLICY mix)
    else:
        p = (s + dtype(min_policy)) / (dtype(1.0) + dtype(min_policy) * a_n)  # NetworkVP_discrate.py:73-74
    if not keep:
        return p, v
    return dict(x=xq, col1=col1, n1=n1, col2=col2, n2=n2, flat=flat, d1=d1, v=v, z=z, s=s, p=p, lsm=zs - np.log(e.sum(axis=1, keepdims=True)),
                w11=w11, w12=w12, w1=w1)


# --------------------------------------------------------------------------------------
# loss + analytic backward (SURVEY Appendix A.3 / A.4)
# --------------------------------------------------------------------------------------
def losses_from_heads(p, v, y_r, a, beta, log_eps, v_stop=None):
    """NetworkVP_discrate.py:61, :75-85, :100 -- all reductions are sums.
    `v_stop` (tests only) freezes the value inside the advantage, emulating tf.stop_gradient
    for finite-difference checks."""
    sel = (p * a).sum(axis=1)
    adv = y_r - (v if v_stop is None else v_stop)
    cost_p_1 = np.log(np.maximum(sel, log_eps)) * adv
    cost_p_2 = -beta * (np.log(np.maximum(p, log_eps)) * p).sum(axis=1)
    cost_p_1_agg, cost_p_2_agg = cost_p_1.sum(), cost_p_2.sum()
    cost_p = -(cost_p_1_agg + cost_p_2_agg)
    cost_v = 0.5 * ((y_r - v) ** 2).sum()
    return dict(cost_p_1=cost_p_1_agg, cost_p_2=cost_p_2_agg, cost_p=cost_p, cost_v=cost_v,
                cost_all=cost_p + cost_v)


def losses_from_log_softmax(lsm, s, v, y_r, a, beta, v_stop=None):
    """Config.USE_LOG_SOFTMAX branch, NetworkVP_discrate.py:64-71: log_softmax instead of log(max(softmax, eps))."""
    adv = y_r - (v if v_stop is None else v_stop)
    cost_p_1_agg = ((lsm * a).sum(axis=1) * adv).sum()
    cost_p_2_agg = (-beta * (lsm * s).sum(axis=1)).sum()
    cost_p = -(cost_p_1_agg + cost_p_2_agg)
    cost_v = 0.5 * ((y_r - v) ** 2).sum()
    return dict(cost_p_1=cost_p_1_agg, cost_p_2=cost_p_2_agg, cost_p=cost_p, cost_v=cost_v, cost_all=cost_p + cost_v)


def loss_and_grads(params, x, y_r, a, *, geom=None, beta=0.01, log_eps=1e-6, min_policy=0.0,
                   dtype=np.float64, quant=None, keep=False, use_log_softmax=False, part="all", v_stop=None):
    """A5 minus the optimizer: returns (losses dict, grads dict keyed like params); with keep=True
    also the forward cache extended by the backward intermediates dd1 / dn2 / dn1 / dz / dv.
    `v_stop` (finite-difference tests only) freezes the value inside the advantage, as in losses_from_heads."""
    g = _geom(geom)
    f = forward(params, x, geom=g, dtype=dtype, quant=quant, min_policy=min_policy, keep=True, use_log_softmax=use_log_softmax)
    b = x.shape[0]
    y_r = np.asarray(y_r, dtype=dtype)
    a = np.asarray(a, dtype=dtype)
    beta = dtype(beta)
    log_eps = dtype(log_eps)
    p, v, s, d1 = f["p"], f["v"], f["s"], f["d1"]
    a_n = p.shape[1]

    # heads backward
    adv = y_r - (v if v_stop is None else v_stop)            # stop_gradient on v here
    dv = v - y_r                                             # from cost_v only
    if use_log_softmax:
        # d/dz of -(sum_a lsm a) adv - (-beta sum lsm s):  -adv (a - s sum(a)) + beta s (lsm - sum(lsm s))
        lsm = f["lsm"]
        losses = losses_from_log_softmax(lsm, s, v, y_r, a, beta, v_stop=v_stop)
        dz = -adv[:, None] * (a - s * a.sum(axis=1, keepdims=True)) + beta * s * (lsm - (lsm * s).sum(axis=1, keepdims=True))
    else:
        losses = losses_from_heads(p, v, y_r, a, beta, log_eps, v_stop=v_stop)
        sel = (p * a).sum(axis=1)
        gz = (-a * ((sel >= log_eps) * adv / np.where(sel >= log_eps, sel, 1))[:, None]
              + beta * (np.log(np.maximum(p, log_eps)) + (p >= log_eps)))
        h = gz / (dtype(1.0) + dtype(min_policy) * a_n)
        dz = s * (h - (s * h).sum(axis=1, keepdims=True))
    # Config.DUAL_RMSPROP minimises cost_p and cost_v separately (NetworkVP_discrate.py:87-98, :124-128): part = "p" is the
    # gradient of cost_p alone (nothing reaches logits_v: stop_gradient), part = "v" that of cost_v alone (nothing reaches logits_p)
    if part == "p":
        dv = np.zeros_like(dv)
    elif part == "v":
        dz = np.zeros_like(dz)
    elif part != "all":
        raise ValueError(part)
    wp = params["logits_p/w:0"].astype(dtype)
    wv = params["logits_v/w:0"].astype(dtype)
    grads = {
        "logits_p/w:0": d1.T @ dz, "logits_p/b:0": dz.sum(axis=0),
        "logits_v/w:0": d1.T @ dv[:, None], "logits_v/b:0": dv.sum(keepdims=True),
    }
    dd1 = (dz @ wp.T + dv[:, None] * wv.T) * (d1 > 0)
    dd1 = _q(dd1, quant, dtype)                              # CUDA stores dd1 as bf16
    grads["dense1/w:0"] = f["flat"].T @ dd1
    grads["dense1/b:0"] = dd1.sum(axis=0)
    dflat = (dd1 @ f["w1"].T) * (f["flat"] > 0)
    dn2 = _q(dflat, quant, dtype).reshape(-1, C2_OUT)
    grads["conv12/w:0"] = f["col2"].T @ dn2
    grads["conv12/b:0"] = dn2.sum(axis=0)
    n_out, lo, hi = zip(same_pad(g.h1, C2_K, C2_S), same_pad(g.w1, C2_K, C2_S))
    dn1 = _col2im(dn2 @ f["w12"].T, b, (g.h1, g.w1), C2_K, C2_S, lo, hi, n_out, C1_OUT) * (f["n1"] > 0)
    dn1 = _q(dn1, quant, dtype).reshape(-1, C1_OUT)
    grads["conv11/w:0"] = f["col1"].T @ dn1
    grads["conv11/b:0"] = dn1.sum(axis=0)
    for k in grads:
        grads[k] = grads[k].reshape(params[k].shape)
    if part != "all":                                        # tf.gradients yields None there: the optimizer skips the variable
        for k in (("logits_v/w:0", "logits_v/b:0") if part == "p" else ("logits_p/w:0", "logits_p/b:0")):
            del grads[k]
    if keep:
        f.update(dd1=dd1, dn2=dn2.reshape(b, -1), dn1=dn1.reshape(b, -1), dz=dz, dv=dv)
        return losses, grads, f
    return losses, grads


# --------------------------------------------------------------------------------------
# RMSProp with TF semantics (SURVEY Appendix A.5) [TF-SEMANTICS]
# --------------------------------------------------------------------------------------
def rmsprop_init(params):
    ms = {k: np.ones_like(v) for k, v in params.items()}     # ms slot starts at 1.0
    mom = {k: np.zeros_like(v) for k, v in params.items()}
    return ms, mom


def rmsprop_update(params, grads, ms, mom, *, lr, rho=0.99, mu=0.0, eps=0.1, dtype=np.float32):
    """In-place on copies; returns (params, ms, mom).  eps is INSIDE the sqrt."""
    new_p, new_ms, new_mom = {}, {}, {}
    for k in params:
        g = grads[k].astype(dtype)
        m = dtype(rho) * ms[k].astype(dtype) + dtype(1.0 - rho) * g * g
        mo = dtype(mu) * mom[k].astype(dtype) + dtype(lr) * g / np.sqrt(m + dtype(eps))
        new_p[k] = (params[k].astype(dtype) - mo)
        new_ms[k], new_mom[k] = m, mo
    return new_p, new_ms, new_mom


def clip_by_average_norm(g, clip_norm):
    """tf.clip_by_average_norm (Config.USE_GRAD_CLIP, NetworkVP_discrate.py:118-121): t * clip / max(||t||_2 / n, clip), n = the
    number of elements of t.  [TF-SEMANTICS]"""
    g = np.asarray(g)
    avg = np.sqrt((g.astype(np.float64) ** 2).sum()) / g.size
    return g * g.dtype.type(clip_norm / max(avg, clip_norm))


def train_step(params, ms, mom, x, y_r, a, *, lr, beta=0.01, log_eps=1e-6, min_policy=0.0, use_log_softmax=False, grad_clip=None,
               rho=0.99, mu=0.0, eps=0.1, dtype=np.float64, quant=None):
    losses, grads = loss_and_grads(params, x, y_r, a, beta=beta, log_eps=log_eps,
                                   min_policy=min_policy, dtype=dtype, quant=quant, use_log_softmax=use_log_softmax)
    applied = grads if grad_clip is None else {k: clip_by_average_norm(g, grad_clip) for k, g in grads.items()}
    p2, ms2, mom2 = rmsprop_update(params, applied, ms, mom, lr=lr, rho=rho, mu=mu, eps=eps, dtype=dtype)
    return losses, grads, p2, ms2, mom2


def clip_by_norm(g, clip_norm):
    """tf.clip_by_norm(g, c) [TF-SEMANTICS]: g * c / max(||g||_2, c)  (NetworkVP_discrate.py:109-110, :114-115)."""
    g = np.asarray(g, dtype=np.float64)
    return g * clip_norm / max(np.sqrt((g * g).sum()), clip_norm)


def train_step_dual(params, slots_p, slots_v, x, y_r, a, *, lr, beta=0.01, log_eps=1e-6, min_policy=0.0, use_log_softmax=False,
                    rho=0.99, mu=0.0, eps=0.1, dtype=np.float64, quant=None, grad_clip=None):
    """Config.DUAL_RMSPROP (NetworkVP_discrate.py:87-98, :124-128): train_op = [minimize(cost_p), minimize(cost_v)], two
    RMSProp optimizers with their own slots.  TensorFlow runs the two train ops of one sess.run in no defined order;
    this restatement takes the order-independent reading [TF-SEMANTICS]: both gradients at the pre-call weights (the forward
    pass is shared in the graph), then w <- w - step_p - step_v.  Variables a cost does not reach are skipped by that
    optimizer (no slot, no decay).  slots_x = (ms, mom) dicts over ALL variables; untouched entries are returned as they came.
    -> (losses, grads_p, grads_v, params', slots_p', slots_v')"""
    kw = dict(beta=beta, log_eps=log_eps, min_policy=min_policy, dtype=dtype, quant=quant, use_log_softmax=use_log_softmax)
    losses, gp = loss_and_grads(params, x, y_r, a, part="p", **kw)
    _, gv = loss_and_grads(params, x, y_r, a, part="v", **kw)
    new_p = {k: v.astype(dtype) for k, v in params.items()}
    out_slots = []
    for g, (ms, mom) in ((gp, slots_p), (gv, slots_v)):
        if grad_clip is not None:       # DUAL_RMSPROP + USE_GRAD_CLIP: clip_by_norm per variable and optimizer (:107-117)
            g = {k: clip_by_norm(v, grad_clip) for k, v in g.items()}
        sub = {k: params[k] for k in g}
        p2, ms2, mom2 = rmsprop_update(sub, g, {k: ms[k] for k in g}, {k: mom[k] for k in g}, lr=lr, rho=rho, mu=mu, eps=eps, dtype=dtype)
        for k in g:
            new_p[k] = new_p[k] - (params[k].astype(dtype) - p2[k])
        nms, nmom = dict(ms), dict(mom)
        nms.update(ms2); nmom.update(mom2)
        out_slots.append((nms, nmom))
    return losses, gp, gv, new_p, out_slots[0], out_slots[1]


# --------------------------------------------------------------------------------------
# returns -- ProcessAgent.py:70-84, restated on plain reward lists (Python floats = fp64)
# --------------------------------------------------------------------------------------
def accumulate_rewards(rewards, discount, terminal_reward, *, discounting=True,
                       use_intermediate_reward=False, reward_clipping=True, rmin=-1.0, rmax=1.0):
    """Returns the list of n rewards after the reference's in-place update.

    Default config: out[t] = gamma^(n-1-t) * terminal for t < n-1, out[n-1] untouched.
    USE_INTERMEDIATE_REWARD=True (ProcessAgent.py:79-80): the running sum is discounted twice
    and experiences[t].reward is never written -- rewards come back unchanged.
    """
    out = [float(r) for r in rewards]
    reward_sum = float(terminal_reward)
    for t in reversed(range(0, len(out) - 1)):
        r = min(max(out[t], rmin), rmax) if reward_clipping else out[t]
        if discounting:
            reward_sum = discount * reward_sum
            if use_intermediate_reward:
                reward_sum = discount * reward_sum + r
            else:
                out[t] = reward_sum
    return out


def nstep_returns(rewards, discount, seed, *, clip=(-1.0, 1.0)):
    """Upstream NVlabs semantics (the commented ProcessAgent.py:83/:146): R_t = clip(r_t) + g*R_{t+1},
    seeded with R_{n-1} := seed, n-1 rows emitted."""
    n = len(rewards)
    out = [0.0] * max(n - 1, 0)
    run = float(seed)
    for t in reversed(range(0, n - 1)):
        r = float(rewards[t])
        if clip is not None:
            r = min(max(r, clip[0]), clip[1])
        run = discount * run + r
        out[t] = run
    return out


# --------------------------------------------------------------------------------------
# sampling -- ProcessAgent.py:110-115 ; np.random.choice(actions, p=p) restated (SURVEY A.6)
# --------------------------------------------------------------------------------------
def select_action(p, u):
    """p: float32/64 [A]; u: one uniform in [0,1) (what random_sample() returned)."""
    cdf = np.cumsum(np.asarray(p, dtype=np.float64))
    cdf /= cdf[-1]
    return int(np.searchsorted(cdf, u, side="right"))


def select_actions(p, u):
    return np.array([select_action(p[i], u[i]) for i in range(len(u))], dtype=np.int32)
