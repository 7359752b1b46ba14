"""CPU tests of the TensorBoard summaries of the MLP networks' log: the histogram tags of the fork NetworkVP and of
NetworkVP_discrate (ga3c_b200.summaries.mlp_histogram_tags) against the variable tables of oracle/oracle_mlp.py, and -- where
$GA3C_REFERENCE names the original sources -- against the tags the reference's own NetworkVP.py / NetworkVP_discrate.py pass
to tf.summary.histogram and tf.summary.scalar."""
import os
import re

import pytest

from oracle import oracle_mlp as om

MAX_SOURCES = 23            # HISTO_MAX_SRC (csrc/kernels.h)


def tags_of(kind, s, a, dense_layers=om.DISCRATE_DENSE_LAYERS):
    from ga3c_b200 import summaries
    shapes = om.param_shapes(kind, s, a, dense_layers)
    dead = set(om.dead_params(kind, dense_layers))
    return summaries.mlp_histogram_tags([(n, n not in dead) for n in shapes])


def expected(kind, s, a, dense_layers=om.DISCRATE_DENSE_LAYERS):
    weights = ["weights_" + n.replace(":", "_") for n in om.param_shapes(kind, s, a, dense_layers)]
    layers = ["activation_" + name for name, _, _ in om.layers_of(kind, dense_layers)]
    return weights + layers + ["activation_v", "activation_p"]


FORK_VP = ["weights_dense11_p/w_0", "weights_dense11_p/b_0", "weights_dense12_p/w_0", "weights_dense12_p/b_0",
           "weights_dense13_p/w_0", "weights_dense13_p/b_0", "weights_dense14_p/w_0", "weights_dense14_p/b_0",
           "weights_dense1/w_0", "weights_dense1/b_0", "weights_logits_v/w_0", "weights_logits_v/b_0",
           "weights_logits_p/out_x/w_0", "weights_logits_p/out_x/b_0", "weights_logits_p/out_y/w_0", "weights_logits_p/out_y/b_0",
           "activation_dense11_p", "activation_dense12_p", "activation_dense13_p", "activation_dense14_p", "activation_dense1",
           "activation_v", "activation_p"]
DISCRATE = ["weights_dense1_1_p/w_0", "weights_dense1_1_p/b_0", "weights_dense1_2_p/w_0", "weights_dense1_2_p/b_0",
            "weights_dense1_3_p/w_0", "weights_dense1_3_p/b_0", "weights_dense1_4_p/w_0", "weights_dense1_4_p/b_0",
            "weights_logits_v/w_0", "weights_logits_v/b_0", "weights_logits_p/w_0", "weights_logits_p/b_0",
            "activation_dense1_4_p", "activation_v", "activation_p"]


@pytest.mark.parametrize("kind,s,a,want", [("fork_vp", 3, 1, FORK_VP), ("fork_vp", 4, 2, FORK_VP), ("discrate", 4, 2, DISCRATE)])
def test_tags_of_the_default_networks(kind, s, a, want):
    got = tags_of(kind, s, a)
    assert got == want == expected(kind, s, a)
    assert len(got) <= MAX_SOURCES and len(set(got)) == len(got)


@pytest.mark.parametrize("n_dense", range(1, 9))
def test_tags_of_discrate_for_every_dense_layers_length(n_dense):
    dense = tuple(10 + 3 * i for i in range(n_dense))
    got = tags_of("discrate", 4, 2, dense)
    assert got == expected("discrate", 4, 2, dense)
    assert len(got) == 2 * n_dense + 4 + 1 + 2 <= MAX_SOURCES           # variables, the one live layer, v, p
    assert [t for t in got if t.startswith("activation_")] == [f"activation_dense1_{n_dense}_p", "activation_v", "activation_p"]


def _summary_literals(path):
    """The first argument of every tf.summary.histogram( / tf.summary.scalar( call in the file, when it is a string literal."""
    text = open(path).read()
    hist = re.findall(r"tf\.summary\.histogram\(\s*(['\"])(.*?)\1", text)
    scal = re.findall(r"tf\.summary\.scalar\(\s*(['\"])(.*?)\1", text)
    return [h for _, h in hist], [s for _, s in scal]


@pytest.mark.reference
@pytest.mark.parametrize("kind,fname", [("fork_vp", "NetworkVP.py"), ("discrate", "NetworkVP_discrate.py")])
def test_tags_cover_the_reference_summaries(kind, fname):
    """Every tag the reference writes is one of ours: histogram literals as they stand, or as a "%s" pattern over the
    variable names (weights_%s); scalar literals among the six scalars."""
    from ga3c_b200 import summaries
    path = os.path.join(os.environ["GA3C_REFERENCE"], fname)
    if not os.path.exists(path):
        pytest.skip(f"{fname} is not in $GA3C_REFERENCE")
    hist, scal = _summary_literals(path)
    ours = tags_of(kind, 4, 2)
    for lit in hist:
        if "%" in lit:
            pat = re.compile(re.escape(lit).replace("%s", ".+").replace("%d", r"\d+") + "$")
            assert any(pat.match(t) for t in ours), (lit, ours)
        else:
            assert summaries.clean_tag(lit) in ours, (lit, ours)
    assert set(scal) <= set(summaries.SCALAR_TAGS), scal
