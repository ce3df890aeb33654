"""SMPL_Dataset (avatarclip_b200/dataset.py) loading the render directories the reference SHIPS
(data/zero_beta_{tpose,standpose}_render) against the reference's own constructor lines (models/dataset.py:204-250): a sample of 4
of each directory's 108 frames (PNGs + transforms_train.json trimmed to those frames) is stored under
tests/golden/shipped_render_sample, and what the reference's lines built from it -- image scaling, the W-axis flip of :222,
masks, poses, focal, K, bounding box; tensors as sha256 of their bytes -- in tests/golden/host_mirrors.json
(oracle/pin_host_mirrors.py)."""
import hashlib
import json
import os

import numpy as np
import pytest
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


class _Conf(dict):
    def get_string(self, k):
        return self[k]


def _sha(t):
    return hashlib.sha256(np.ascontiguousarray(t.detach().cpu().numpy()).tobytes()).hexdigest()


@pytest.mark.parametrize("name", ["zero_beta_tpose_render", "zero_beta_standpose_render"])
def test_shipped_render_directory_loads_like_the_reference(name):
    from avatarclip_b200.dataset import SMPL_Dataset
    data_dir = os.path.join(GOLDEN, "shipped_render_sample", name)
    ref = json.load(open(os.path.join(GOLDEN, "host_mirrors.json")))["dataset"][name]
    ours = SMPL_Dataset(_Conf(data_dir=data_dir), device="cpu")
    assert ours.n_images == ref["n_images"] == 4 and (ours.H, ours.W) == (ref["H"], ref["W"]) == (256, 256)
    assert ours.focal == ref["focal"] and ours.image_pixels == ref["image_pixels"]
    for k in ("images", "masks", "poses", "K"):
        t = getattr(ours, k)
        assert list(t.shape) == ref["shapes"][k] and _sha(t) == ref[k], k
    assert ours.images.dtype == ours.masks.dtype == ours.poses.dtype == torch.float32 and ours.K.dtype == torch.float64
    assert np.array_equal(ours.object_bbox_min, ref["object_bbox_min"]) and np.array_equal(ours.object_bbox_max, ref["object_bbox_max"])
    assert [os.path.relpath(p, data_dir) for p in ours.images_lis] == ref["images_lis"]
    img = ours.image_at(2, 4)                                    # frame 58 of the shipped directory: train_clip's validation camera (main.py:557)
    assert img.shape == (64, 64, 3)
