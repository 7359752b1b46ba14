"""The conv NetworkVP oracle for any input geometry (Config.IMAGE_HEIGHT, IMAGE_WIDTH, STACKED_FRAMES): the arithmetic of
oracle/oracle_np.py (same modes, same bf16 rounding points, same heads, loss and backward) with H, W, C as arguments and
non-square frames.  TEST INFRASTRUCTURE ONLY.  oracle_np keeps its fixed 84x84x4 module constants, which its golden files and
tests pin; at 84x84x4 this module computes what oracle_np does (test_geometry.py checks it)."""
from __future__ import annotations

import numpy as np

from oracle import oracle_np as onp

C1_K, C1_S, C1_OUT = onp.C1_K, onp.C1_S, onp.C1_OUT
C2_K, C2_S, C2_OUT = onp.C2_K, onp.C2_S, onp.C2_OUT
FC = onp.FC


class Geometry:
    """Derived sizes of input (h, w, c) under TF SAME padding (SURVEY A.1)."""

    def __init__(self, h: int, w: int, c: int):
        self.h, self.w, self.c = h, w, c
        self.h1, self.pt1, _ = onp.same_pad(h, C1_K, C1_S)
        self.w1, self.pl1, _ = onp.same_pad(w, C1_K, C1_S)
        self.h2, self.pt2, _ = onp.same_pad(self.h1, C2_K, C2_S)
        self.w2, self.pl2, _ = onp.same_pad(self.w1, C2_K, C2_S)
        self.state_dim = h * w * c
        self.flat = self.h2 * self.w2 * C2_OUT

    def __repr__(self):
        return f"{self.h}x{self.w}x{self.c}"


def param_shapes(g: Geometry, num_actions: int):
    s = onp.param_shapes(num_actions)
    s["conv11/w:0"] = (C1_K, C1_K, g.c, C1_OUT)
    s["dense1/w:0"] = (g.flat, FC)
    return s


def init_params(rng, g: Geometry, num_actions: int = 6):
    fan_in = {"conv11": C1_K * C1_K * g.c, "conv12": C2_K * C2_K * C1_OUT, "dense1": g.flat, "logits_v": FC, "logits_p": FC}
    return {k: rng.uniform(-1 / np.sqrt(fan_in[k.split("/")[0]]), 1 / np.sqrt(fan_in[k.split("/")[0]]), size=s).astype(np.float32)
            for k, s in param_shapes(g, num_actions).items()}


def synth_frames_u8(rng, g: Geometry, batch: int):
    return rng.integers(0, 256, size=(batch, g.state_dim), dtype=np.uint8)


def normalise(k):
    return (k.astype(np.float32) / np.float32(128.0) - np.float32(1.0)).astype(np.float32)


def _pads(n_in, n_out, k, s):
    total = max((n_out - 1) * s + k - n_in, 0)
    return total // 2, total - total // 2


def im2col(x, k, s, oh, ow):
    """x [B, H, W, C] -> [B*oh*ow, k*k*C], columns (kh, kw, c), TF SAME zero padding (low side smaller)."""
    b, h, w, c = x.shape
    (t, bo), (l, r) = _pads(h, oh, k, s), _pads(w, ow, k, s)
    xp = np.zeros((b, h + t + bo, w + l + r, c), dtype=x.dtype)
    xp[:, t:t + h, l:l + w, :] = x
    sb, sh, sw, sc = xp.strides
    cols = np.lib.stride_tricks.as_strided(xp, shape=(b, oh, ow, k, k, c), strides=(sb, sh * s, sw * s, sh, sw, sc),
                                           writeable=False)
    return cols.reshape(b * oh * ow, k * k * c)


def col2im(dcols, b, h, w, k, s, oh, ow, c):
    (t, bo), (l, r) = _pads(h, oh, k, s), _pads(w, ow, k, s)
    dxp = np.zeros((b, h + t + bo + s, w + l + r + s, c), dtype=dcols.dtype)
    d6 = dcols.reshape(b, oh, ow, k, k, c)
    for kh in range(k):
        for kw in range(k):
            dxp[:, kh:kh + s * oh:s, kw:kw + s * ow:s, :] += d6[:, :, :, kh, kw, :]
    return dxp[:, t:t + h, l:l + w, :]


def forward(g: Geometry, params, x, *, dtype=np.float64, quant=None, min_policy=0.0, keep=False, use_log_softmax=False):
    q = onp._q
    b = x.shape[0]
    xq = q(np.asarray(x, np.float32).reshape(b, g.h, g.w, g.c), quant, dtype)
    w11 = q(params["conv11/w:0"], quant, dtype).reshape(-1, C1_OUT)
    w12 = q(params["conv12/w:0"], quant, dtype).reshape(-1, C2_OUT)
    w1 = q(params["dense1/w:0"], quant, dtype)
    col1 = im2col(xq, C1_K, C1_S, g.h1, g.w1)
    n1 = q(np.maximum(col1 @ w11 + params["conv11/b:0"].astype(dtype), 0), quant, dtype).reshape(b, g.h1, g.w1, C1_OUT)
    col2 = im2col(n1, C2_K, C2_S, g.h2, g.w2)
    n2 = q(np.maximum(col2 @ w12 + params["conv12/b:0"].astype(dtype), 0), quant, dtype)
    flat = n2.reshape(b, g.flat)
    d1 = np.maximum(flat @ w1 + params["dense1/b:0"].astype(dtype), 0)
    v = (d1 @ params["logits_v/w:0"].astype(dtype) + params["logits_v/b:0"].astype(dtype))[:, 0]
    z = d1 @ params["logits_p/w:0"].astype(dtype) + params["logits_p/b:0"].astype(dtype)
    zs = z - z.max(axis=1, keepdims=True)
    e = np.exp(zs)
    s = e / e.sum(axis=1, keepdims=True)
    p = s if use_log_softmax else (s + dtype(min_policy)) / (dtype(1.0) + dtype(min_policy) * z.shape[1])
    if not keep:
        return p, v
    return dict(x=xq, col1=col1, n1=n1, col2=col2, n2=n2, flat=flat, d1=d1, v=v, z=z, s=s, p=p,
                lsm=zs - np.log(e.sum(axis=1, keepdims=True)), w11=w11, w12=w12, w1=w1)


def loss_and_grads(g: Geometry, params, x, y_r, a, *, beta=0.01, log_eps=1e-6, min_policy=0.0, dtype=np.float64, quant=None,
                   keep=False, use_log_softmax=False, part="all", v_stop=None):
    """oracle_np.loss_and_grads for geometry g; v_stop (finite differences only) freezes v inside the advantage."""
    f = forward(g, params, x, dtype=dtype, quant=quant, min_policy=min_policy, keep=True, use_log_softmax=use_log_softmax)
    b = x.shape[0]
    y_r, a = np.asarray(y_r, dtype=dtype), np.asarray(a, dtype=dtype)
    beta, log_eps = dtype(beta), dtype(log_eps)
    p, v, s, d1 = f["p"], f["v"], f["s"], f["d1"]
    vs = v if v_stop is None else v_stop
    if use_log_softmax:
        losses = onp.losses_from_log_softmax(f["lsm"], s, v, y_r, a, beta, v_stop=v_stop)
        adv = y_r - vs
        lsm = f["lsm"]
        dz = -adv[:, None] * (a - s * a.sum(axis=1, keepdims=True)) + beta * s * (lsm - (lsm * s).sum(axis=1, keepdims=True))
    else:
        losses = onp.losses_from_heads(p, v, y_r, a, beta, log_eps, v_stop=v_stop)
        sel = (p * a).sum(axis=1)
        adv = y_r - vs
        gz = (-a * ((sel >= log_eps) * adv / np.where(sel >= log_eps, sel, 1))[:, None]
              + beta * (np.log(np.maximum(p, log_eps)) + (p >= log_eps)))
        h = gz / (dtype(1.0) + dtype(min_policy) * p.shape[1])
        dz = s * (h - (s * h).sum(axis=1, keepdims=True))
    dv = v - y_r
    if part == "p":
        dv = np.zeros_like(dv)
    elif part == "v":
        dz = np.zeros_like(dz)
    wp, wv = params["logits_p/w:0"].astype(dtype), params["logits_v/w:0"].astype(dtype)
    grads = {"logits_p/w:0": d1.T @ dz, "logits_p/b:0": dz.sum(axis=0),
             "logits_v/w:0": d1.T @ dv[:, None], "logits_v/b:0": dv.sum(keepdims=True)}
    dd1 = onp._q((dz @ wp.T + dv[:, None] * wv.T) * (d1 > 0), quant, dtype)
    grads["dense1/w:0"] = f["flat"].T @ dd1
    grads["dense1/b:0"] = dd1.sum(axis=0)
    dn2 = onp._q((dd1 @ f["w1"].T) * (f["flat"] > 0), quant, dtype).reshape(-1, C2_OUT)
    grads["conv12/w:0"] = f["col2"].T @ dn2
    grads["conv12/b:0"] = dn2.sum(axis=0)
    dn1 = col2im(dn2 @ f["w12"].T, b, g.h1, g.w1, C2_K, C2_S, g.h2, g.w2, C1_OUT) * (f["n1"] > 0)
    dn1 = onp._q(dn1, quant, dtype).reshape(-1, C1_OUT)
    grads["conv11/w:0"] = f["col1"].T @ dn1
    grads["conv11/b:0"] = dn1.sum(axis=0)
    grads = {k: v_.reshape(params[k].shape) for k, v_ in grads.items()}
    if part != "all":
        for k in (("logits_v/w:0", "logits_v/b:0") if part == "p" else ("logits_p/w:0", "logits_p/b:0")):
            del grads[k]
    if keep:
        f.update(dd1=dd1, dn2=dn2.reshape(b, -1), dn1=dn1.reshape(b, -1))
        return losses, grads, f
    return losses, grads
