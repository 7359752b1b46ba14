"""CPU checks of the input-geometry support (Config.IMAGE_HEIGHT, IMAGE_WIDTH, STACKED_FRAMES): the geometry-parameterised
oracle (tests/_geometry_oracle.py) against finite differences, torch and oracle_np, and the C ABI's ga3c_config mirror."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from oracle import oracle_np as onp
import _geometry_oracle as go

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _case(g, b, seed=7, num_actions=5):
    rng = np.random.default_rng(seed)
    params = go.init_params(rng, g, num_actions)
    x = go.normalise(go.synth_frames_u8(rng, g, b))
    y_r, a = onp.synth_targets(rng, b, num_actions)
    return params, x, y_r, a


@pytest.mark.parametrize("hwc", [(13, 9, 1), (10, 17, 3)])
def test_oracle_backward_matches_finite_differences(hwc):
    """Non-square, one with C = 1: the analytic fp64 gradients of cost_all against central differences, on a sample of entries
    of every variable (v held fixed inside the advantage, as tf.stop_gradient does)."""
    g = go.Geometry(*hwc)
    params, x, y_r, a = _case(g, 3)
    params = {k: v.astype(np.float64) for k, v in params.items()}
    _, grads, f = go.loss_and_grads(g, params, x, y_r, a, keep=True)
    v_stop = f["v"]
    rng = np.random.default_rng(1)
    eps = 1e-6
    for name, val in params.items():
        for idx in [tuple(rng.integers(0, s) for s in val.shape) for _ in range(6)]:
            hi, lo = {**params}, {**params}
            hi[name] = val.copy(); hi[name][idx] += eps
            lo[name] = val.copy(); lo[name][idx] -= eps
            lh, _ = go.loss_and_grads(g, hi, x, y_r, a, v_stop=v_stop)
            ll, _ = go.loss_and_grads(g, lo, x, y_r, a, v_stop=v_stop)
            num = (lh["cost_all"] - ll["cost_all"]) / (2 * eps)
            assert abs(num - grads[name][idx]) <= 1e-6 + 1e-5 * abs(num), (name, idx, num, grads[name][idx])


@pytest.mark.parametrize("hwc", [(7, 5, 2), (13, 11, 1), (21, 9, 3), (1, 1, 1)])
def test_same_padding_matches_torch_conv2d_after_explicit_pad(hwc):
    """SAME padding split low-side-smaller at odd sizes: both convs of the oracle equal torch conv2d on the explicitly padded
    input (F.pad with the (before, after) split TF uses)."""
    torch = pytest.importorskip("torch")
    F = torch.nn.functional
    g = go.Geometry(*hwc)
    params, x, _, _ = _case(g, 2)
    f = go.forward(g, params, x, keep=True)

    def conv(inp, w, b, k, s):
        _, _, h, wd = inp.shape
        oh, ow = -(-h // s), -(-wd // s)
        ph, pw = max((oh - 1) * s + k - h, 0), max((ow - 1) * s + k - wd, 0)
        inp = F.pad(inp, (pw // 2, pw - pw // 2, ph // 2, ph - ph // 2))
        return torch.relu(F.conv2d(inp, torch.as_tensor(w).permute(3, 2, 0, 1), torch.as_tensor(b), stride=s))

    xt = torch.as_tensor(x.astype(np.float64).reshape(2, g.h, g.w, g.c)).permute(0, 3, 1, 2)
    n1 = conv(xt, params["conv11/w:0"].astype(np.float64), params["conv11/b:0"].astype(np.float64), 8, 4)
    n2 = conv(n1, params["conv12/w:0"].astype(np.float64), params["conv12/b:0"].astype(np.float64), 4, 2)
    assert n1.shape[2:] == (g.h1, g.w1) and n2.shape[2:] == (g.h2, g.w2)
    np.testing.assert_allclose(f["n1"], n1.permute(0, 2, 3, 1).numpy(), rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(f["n2"].reshape(2, g.h2, g.w2, 32), n2.permute(0, 2, 3, 1).numpy(), rtol=1e-12, atol=1e-12)


def test_oracle_equals_oracle_np_at_84x84x4():
    """At the default geometry the parameterised oracle computes what oracle_np does, bf16 mode included."""
    g = go.Geometry(84, 84, 4)
    rng = np.random.default_rng(3)
    params = onp.init_params(rng, 6)
    x = onp.synth_frames(rng, 2)
    y_r, a = onp.synth_targets(rng, 2, 6)
    for quant in (None, "bf16"):
        l1, g1 = onp.loss_and_grads(params, x, y_r, a, quant=quant)
        l2, g2 = go.loss_and_grads(g, params, x, y_r, a, quant=quant)
        for k in l1:
            assert l1[k] == pytest.approx(l2[k], rel=1e-12)
        for k in g1:
            np.testing.assert_allclose(g2[k], g1[k], rtol=1e-10, atol=1e-12)


@pytest.mark.parametrize("h,w,c", [(1, 1, 1), (256, 256, 8), (1, 256, 1), (256, 1, 8), (84, 84, 4), (105, 80, 4), (100, 100, 2)])
def test_derived_sizes_follow_the_formula(h, w, c):
    """H1 = ceil(H/4), H2 = ceil(H1/2) (likewise W), K = H2*W2*32, at the ends of the accepted range; padding low side smaller."""
    g = go.Geometry(h, w, c)
    assert (g.h1, g.w1) == (-(-h // 4), -(-w // 4))
    assert (g.h2, g.w2) == (-(-g.h1 // 2), -(-g.w1 // 2))
    assert g.flat == g.h2 * g.w2 * 32
    for n, o, k, s, lo in ((h, g.h1, 8, 4, g.pt1), (w, g.w1, 8, 4, g.pl1), (g.h1, g.h2, 4, 2, g.pt2)):
        total = max((o - 1) * s + k - n, 0)
        assert lo == total // 2 and lo <= total - lo
    if (h, w, c) == (84, 84, 4):
        assert (g.h1, g.h2, g.flat) == (onp.H1, onp.H2, onp.FLAT)
    if (h, w) == (100, 100):
        assert (g.h2 * g.w2) % 2 == 1 and g.flat % 64 != 0        # K not a multiple of the GEMM's 64-wide k-block
    if (h, w) == (256, 256):
        assert g.flat == 32 * 32 * 32


def _header_struct_layout():
    """Field names of ga3c_config, in order, parsed from the header."""
    text = open(os.path.join(ROOT, "include", "ga3c_b200.h")).read()
    body = re.search(r"typedef struct ga3c_config \{(.*?)\} ga3c_config;", text, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    return re.findall(r"(int32_t|float)\s+(\w+);", body)


def test_config_mirror_matches_the_header():
    """The ctypes ga3c_config has the header's fields in the header's order and types; the geometry fields are the last three."""
    from ga3c_b200 import _capi
    fields = _header_struct_layout()
    mirror = [(n, t) for n, t in _capi.ga3c_config._fields_]
    assert [n for _, n in fields] == [n for n, _ in mirror]
    for (ct, name), (_, t) in zip(fields, mirror):
        assert t is (C.c_int32 if ct == "int32_t" else C.c_float), name
    assert [n for _, n in fields[-3:]] == ["image_height", "image_width", "stacked_frames"]
    assert C.sizeof(_capi.ga3c_config) == 4 * len(fields)


def test_header_compiles_as_c99_and_reports_the_struct_size(tmp_path):
    """The header is plain C99; compiled by a C compiler, sizeof(ga3c_config) equals the ctypes mirror's and the geometry fields
    sit at its end."""
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no C compiler")
    from ga3c_b200 import _capi
    src = tmp_path / "t.c"
    src.write_text('#include "ga3c_b200.h"\n#include <stdio.h>\n#include <stddef.h>\n'
                   'int main(void) { printf("%zu %zu\\n", sizeof(ga3c_config), offsetof(ga3c_config, stacked_frames)); return 0; }\n')
    exe = tmp_path / "t"
    subprocess.run([cc, "-std=c99", "-Wall", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                   check=True)
    size, off = map(int, subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split())
    assert size == C.sizeof(_capi.ga3c_config)
    assert off == _capi.ga3c_config.stacked_frames.offset == size - 4


@pytest.mark.parametrize("knob,value", [("IMAGE_HEIGHT", 0), ("IMAGE_HEIGHT", 257), ("IMAGE_WIDTH", 0), ("IMAGE_WIDTH", -3),
                                        ("STACKED_FRAMES", 0), ("STACKED_FRAMES", 9)])
def test_geometry_knobs_out_of_range_are_named(knob, value):
    """Network's reading of the three knobs refuses a value outside 1..256 / 1..8 by name (before any device work), so a 0 never
    reaches the C struct, where it means the default."""
    from ga3c_b200.config import Config
    from ga3c_b200.network import geometry

    class Cfg(Config):
        pass
    setattr(Cfg, knob, value)
    with pytest.raises(ValueError, match=knob):
        geometry(Cfg)
    assert geometry(Config) == (84, 84, 4)
