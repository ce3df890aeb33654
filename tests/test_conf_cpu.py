"""HOCON-subset reader: accessor API of pyhocon's ConfigTree as the reference uses it (main.py:39-127)."""
import glob
import os
import tarfile

import pytest

from avatarclip_b200 import conf

SHIPPED = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "shipped_confs.tar.xz")


@pytest.fixture(scope="module")
def shipped_confs(tmp_path_factory):
    """The reference's confs/ tree as it ships (180 files, stored verbatim in tests/golden by oracle/pin_host_mirrors.py)."""
    d = tmp_path_factory.mktemp("shipped")
    with tarfile.open(SHIPPED) as tf:
        tf.extractall(d, filter="data")
    return str(d)

SAMPLE = """
general {
    base_exp_dir = ./exp/smpl/demo     # trailing comment
    recording = [
        ./,
        ./models
    ]
}
train { learning_rate = 5e-4, end_iter = 100000, use_white_bkgd = False
        warm_up_end = 500 }
clip {
    prompt = a 3D rendering of a {TOREPLACE} in unreal engine
}
model {
    nerf {
        D = 4,
        skips=[4],
        use_viewdirs=True
    }
    sdf_network { d_out = 257, skip_in = [4], scale = 1.0, weight_norm = True }
}
"""


def test_sample():
    c = conf.parse_string(SAMPLE)
    assert c["general.base_exp_dir"] == "./exp/smpl/demo"
    assert c["general.recording"] == ["./", "./models"]
    assert c.get_float("train.learning_rate") == 5e-4 and c.get_int("train.end_iter") == 100000
    assert c.get_bool("train.use_white_bkgd") is False
    assert c.get_float("train.anneal_end", default=0.0) == 0.0
    assert c.get_string("clip.prompt") == "a 3D rendering of a {TOREPLACE} in unreal engine"
    assert dict(c["model.sdf_network"]) == {"d_out": 257, "skip_in": [4], "scale": 1.0, "weight_norm": True}
    assert c["model.nerf.D"] == 4 and c["model.nerf"]["use_viewdirs"] is True
    with pytest.raises(conf.ConfigMissingException):
        c.get_float("train.clip_weight")
    with pytest.raises(KeyError):        # the reference catches bare `except:` / KeyError (main.py:67-127)
        c["dataset.template_obj"]


def test_all_shipped_confs_parse(shipped_confs):
    files = glob.glob(os.path.join(shipped_confs, "confs/**/*.conf"), recursive=True)
    assert len(files) == 180
    for f in files:
        c = conf.parse_file(f)
        kw = dict(c["model.sdf_network"])
        assert kw["d_out"] in (257, 129) and isinstance(kw["skip_in"], list)
        assert {"n_samples", "n_importance", "n_outside", "up_sample_steps", "perturb"} <= set(c["model.neus_renderer"].keys())
        assert c.get_float("train.learning_rate") > 0


def test_every_shipped_conf_constructs_its_networks_and_is_a_supported_loop(shipped_confs):
    """All 180 shipped confs: the model subtrees are accepted as constructor kwargs (main.py:137-151) -- 3 distinct network
    configurations, incl. the extra_color-less one of base_models/astrongman.conf -- and the train.* switches name a loop the
    Runner implements (train_clip: use_silhouettes + extra_color; --mode train: astrongman.conf)."""
    import json
    import avatarclip_b200 as ab
    files = sorted(glob.glob(os.path.join(shipped_confs, "confs/**/*.conf"), recursive=True))
    built, n_clip = {}, 0
    for f in files:
        c = conf.parse_file(f)
        key = json.dumps({k: dict(c["model." + k]) for k in ("sdf_network", "variance_network", "rendering_network",
                                                              "neus_renderer")}, sort_keys=True)
        if key not in built:
            sdf = ab.SDFNetwork(**c["model.sdf_network"])
            var = ab.SingleVarianceNetwork(**c["model.variance_network"])
            col = ab.RenderingNetwork(**c["model.rendering_network"])
            built[key] = ab.NeuSRenderer(None, sdf, var, col, **c["model.neus_renderer"])
        ren = built[key]
        if c.get_bool("train.use_silhouettes", default=False):            # a train_clip conf (main.py:337-566)
            n_clip += 1
            assert ren.extra_color and c.get_bool("model.rendering_network.extra_color", default=False)
            assert c.get_float("train.clip_weight", default=None) is not None and c.get_string("clip.prompt")
        else:                                                              # the NeuS pre-fit conf (main.py:180-256)
            assert f.endswith("base_models/astrongman.conf") and not ren.extra_color
    assert len(built) == 3 and n_clip == 179
