"""Network modules against the UNMODIFIED reference modules (models/{embedder,fields}.py): same parameters under the same torch
seed (the geometric initialisation of models/fields.py:40-63 and nn.Linear's default draws, in the same order), same state-dict
keys in the same order, checkpoints interchangeable in both directions -- for the train_clip networks (extra_color = True) and
for the network of confs/base_models/astrongman.conf (--mode train, no extra head).  The reference side (keys, shapes, sha256
of every tensor, the generator's next draw) was recorded by oracle/pin_host_mirrors.py into tests/golden/host_mirrors.json."""
import hashlib
import json
import os

import numpy as np
import pytest
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SDF_S = dict(d_in=3, d_out=257, d_hidden=256, n_layers=4, skip_in=[4], multires=6, bias=0.5, scale=1.0,
             geometric_init=True, weight_norm=True)
SDF_B2 = dict(SDF_S, n_layers=8)
SDF_SMALL = dict(SDF_S, d_out=129, d_hidden=128, n_layers=3, skip_in=[3])
COL = dict(d_feature=256, mode="no_view_dir", d_in=6, d_out=3, d_hidden=256, n_layers=2, weight_norm=True, multires_view=0,
           squeeze_out=True)


def _ref(name):
    return json.load(open(os.path.join(GOLDEN, "host_mirrors.json")))["fields"][name]


def _sha(t):
    return hashlib.sha256(np.ascontiguousarray(t.detach().cpu().numpy()).tobytes()).hexdigest()


def _build(our_cls, kw, seed):
    torch.manual_seed(seed)
    ours = our_cls(**kw)
    return ours, float(torch.rand(1))


def _same_state(ref, ours):
    b = ours.state_dict()
    assert list(b.keys()) == ref["keys"]
    assert [list(v.shape) for v in b.values()] == ref["shapes"]
    for k, v, h in zip(b.keys(), b.values(), ref["sha256"]):
        assert _sha(v) == h, k
    assert [n for n, _ in ours.named_parameters()] == ref["param_names"]      # torch.optim order
    ours.load_state_dict(b)           # strict: the reference's state dict has exactly these keys and shapes


@pytest.mark.parametrize("kw", [SDF_S, SDF_B2, SDF_SMALL], ids=["shipped", "b2", "small"])
def test_sdf_network_init_is_bit_identical(kw, request):
    import avatarclip_b200 as ab
    ref = _ref("sdf_" + request.node.callspec.id)
    ours, after_ours = _build(ab.SDFNetwork, kw, 0)
    assert after_ours == ref["rand_after"], "the constructor must consume torch's generator exactly like the reference's"
    _same_state(ref, ours)


@pytest.mark.parametrize("extra_color", [True, False])
def test_rendering_network_init_is_bit_identical(extra_color):
    import avatarclip_b200 as ab
    ref = _ref("col_extra" if extra_color else "col_plain")
    ours, after_ours = _build(ab.RenderingNetwork, dict(COL, extra_color=extra_color), 3)
    assert after_ours == ref["rand_after"], "the constructor must consume torch's generator exactly like the reference's"
    _same_state(ref, ours)
    assert hasattr(ours, "extra_lin") == extra_color == ref["has_extra_lin"]


def test_variance_network_and_renderer_constructor():
    import avatarclip_b200 as ab
    _same_state(_ref("variance"), ab.SingleVarianceNetwork(0.3))
    sdf, col, var = ab.SDFNetwork(**SDF_SMALL), ab.RenderingNetwork(**dict(COL, d_feature=128, d_hidden=128)), \
        ab.SingleVarianceNetwork(0.3)
    ren = ab.NeuSRenderer(None, sdf, var, col, n_samples=32, n_importance=32, n_outside=0, up_sample_steps=4, perturb=1.0)
    assert ren.extra_color is False          # the astrongman.conf renderer block: no extra_color key (renderer.py:83)
    with pytest.raises(ValueError):          # 6-channel colour net under a 3-channel renderer (renderer.py:227-232)
        ab.NeuSRenderer(None, sdf, var, ab.RenderingNetwork(**dict(COL, d_feature=128, d_hidden=128, extra_color=True)),
                        32, 32, 0, 4, 1.0)
    with pytest.raises(NotImplementedError):
        ab.NeuSRenderer(None, sdf, var, col, 32, 32, 8, 4, 1.0)       # n_outside > 0: NeRF background, dead in every conf
