"""Runner.validate_image's host side (batching, normal-image rotation, scaling, file names, image layout) against the reference's
own method text (main.py:741-820), both driven by the SAME fake dataset and the SAME fake renderer (deterministic functions of
the rays, CPU tensors) -- the render itself is covered by the GPU parity tests.  The reference side was recorded by executing
the methods in place on these fakes (oracle/pin_host_mirrors.py -> tests/golden/host_mirrors.{json,npz})."""
import json
import os

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden")


def _golden():
    return json.load(open(os.path.join(GOLDEN, "host_mirrors.json"))), np.load(os.path.join(GOLDEN, "host_mirrors.npz"))


class FakeDataset:
    n_images, H, W = 5, 24, 24

    def __init__(self):
        g = torch.Generator().manual_seed(3)
        q, _ = torch.linalg.qr(torch.randn(5, 3, 3, generator=g))
        self.poses = torch.eye(4).repeat(5, 1, 1)
        self.poses[:, :3, :3] = q
        self.poses[:, :3, 3] = torch.randn(5, 3, generator=g)

    def gen_rays_at(self, idx, resolution_level=1):
        n = self.H // resolution_level
        yy, xx = torch.meshgrid(torch.linspace(-1, 1, n), torch.linspace(-1, 1, n), indexing="ij")
        d = torch.stack([xx, -yy, -torch.ones_like(xx)], -1)
        d = d / d.norm(dim=-1, keepdim=True)
        d = torch.sum(d[..., None, :] * self.poses[idx, :3, :3], -1)
        return self.poses[idx, None, None, :3, 3].expand(d.shape), d

    def near_far_from_sphere(self, o, d, is_sphere=False):
        return torch.zeros(o.shape[0], 1), torch.ones(o.shape[0], 1) * 2

    def image_at(self, idx, resolution_level):
        n = self.H // resolution_level
        return ((np.arange(n * n * 3).reshape(n, n, 3) * 7 + idx) % 256).astype(np.uint8)


class FakeRenderer:
    n_samples, n_importance = 3, 2

    def render(self, rays_o, rays_d, near, far, cos_anneal_ratio=0.0, background_rgb=None, **kw):
        S = 5
        k = torch.arange(1, S + 1, dtype=torch.float32)
        w = torch.softmax(rays_d[:, :1] * k[None], dim=1)
        return {"color_fine": torch.sigmoid(rays_d * 3 + rays_o),
                "extra_color_fine": torch.sigmoid(rays_d * -2 + 0.3) * 1.3,                 # > 1 in places: exercises the clip
                "gradients": torch.sin(rays_d[:, None, :] * k[None, :, None]), "weights": w,
                "inside_sphere": (torch.arange(S) % 2).float()[None].expand(rays_d.shape[0], S),
                "weight_sum": w.sum(1, keepdim=True), "mid_z_vals": w}


@pytest.mark.parametrize("extra_color", [True, False])
def test_validate_image_files_equal_the_reference_methods(tmp_path, extra_color):
    import cv2 as cv
    from avatarclip_b200.runner import Runner
    conf = open(os.path.join(HERE, "runner_conf_sample.conf")).read().replace("./exp/CASE_NAME/demo", str(tmp_path / "ours"))
    if not extra_color:
        conf = conf.replace("        extra_color = True\n", "")
    p = tmp_path / "c.conf"
    p.write_text(conf)
    r = Runner(str(p), mode="validate", case="smpl", device="cpu")
    r.dataset, r.iter_step, r.batch_size = FakeDataset(), 1234, 100              # 144 rays at level 2: two uneven batches
    r.renderer.render = FakeRenderer().render
    r.renderer.n_samples, r.renderer.n_importance = 3, 2
    img, extra, normal = r.validate_image(idx=3, resolution_level=2)
    meta, arrays = _golden()
    ref_files = meta["validate_image"][str(int(extra_color))]
    name = "00001234_0_3.png"
    assert {d: sorted(os.listdir(os.path.join(str(tmp_path / "ours"), d))) for d in ref_files} == ref_files
    for d in ("validations_fine", "normals") + (("validations_extra_fine",) if extra_color else ()):
        a = cv.imread(os.path.join(str(tmp_path / "ours"), d, name), cv.IMREAD_UNCHANGED)
        b = arrays[f"validate_image_{int(extra_color)}/{d}/{name}"]
        assert a is not None and a.shape == b.shape and np.array_equal(a, b), d
    assert img.shape == (12, 12, 3) and normal.shape == (12, 12, 3) and (extra is None) == (not extra_color)
    if not extra_color:                       # the reference creates the directory but writes nothing into it
        assert os.listdir(os.path.join(str(tmp_path / "ours"), "validations_extra_fine")) == []


class MeshRenderer(FakeRenderer):
    def __init__(self):
        g = torch.Generator().manual_seed(5)
        self.vertices = (torch.rand(257, 3, generator=g, dtype=torch.float64) - 0.5).numpy()
        self.triangles = torch.randint(0, 257, (300, 3), generator=g).numpy()

    def extract_geometry(self, bound_min, bound_max, resolution, threshold=0.0):
        return self.vertices, self.triangles

    def render(self, rays_o, rays_d, near, far, cos_anneal_ratio=0.0, background_rgb=None, **kw):
        out = super().render(rays_o, rays_d, near, far)
        # view-dependent depth: which of the six views "sees" a vertex best differs from vertex to vertex
        out["mid_z_vals"] = (rays_o.norm(dim=-1, keepdim=True) + torch.cos(rays_d[:, :1] * 9 + rays_o[:, 1:2])).expand(-1, 5)
        return out


@pytest.mark.parametrize("extra_color", [True, False])
def test_validate_mesh_colours_equal_the_reference_methods(tmp_path, extra_color):
    from avatarclip_b200.handoff import read_ply
    from avatarclip_b200.runner import Runner
    conf = open(os.path.join(HERE, "runner_conf_sample.conf")).read().replace("./exp/CASE_NAME/demo", str(tmp_path / "ours"))
    if not extra_color:
        conf = conf.replace("        extra_color = True\n", "")
    p = tmp_path / "c.conf"
    p.write_text(conf)
    r = Runner(str(p), mode="validate", case="smpl", device="cpu")
    r.dataset, r.iter_step, r.batch_size = FakeDataset(), 77, 100               # 257 vertices: three uneven batches per view
    r.dataset.object_bbox_min, r.dataset.object_bbox_max = np.array([-1.01] * 3), np.array([1.01] * 3)
    mr = MeshRenderer()
    r.renderer.render, r.renderer.extract_geometry = mr.render, mr.extract_geometry
    path = r.validate_mesh(resolution=64)
    meta, arrays = _golden()
    captured = dict(meta["validate_mesh"][str(int(extra_color))],
                    **{k: arrays[f"validate_mesh_{int(extra_color)}_{k}"] for k in ("vertices", "triangles", "colors")})
    v, f, c = read_ply(path)
    assert os.path.basename(path) == os.path.basename(captured["path"]) == "00000077.ply" and captured["file_type"] == "ply"
    assert np.array_equal(f, captured["triangles"].astype(np.int32)) and np.allclose(v, captured["vertices"].astype(np.float32))
    assert c.shape == captured["colors"].shape == (257, 3)
    assert np.array_equal(c, captured["colors"])                 # the same view wins for every vertex, the same 8-bit colour


class CastLightDataset(FakeDataset):
    def gen_rays_pose(self, pose, resolution_level=1):
        pose = torch.as_tensor(np.asarray(pose), dtype=torch.float32)
        n = int(self.H // resolution_level)
        yy, xx = torch.meshgrid(torch.linspace(-1, 1, n), torch.linspace(-1, 1, n), indexing="ij")
        d = torch.stack([xx, -yy, -torch.ones_like(xx)], -1)
        d = d / d.norm(dim=-1, keepdim=True)
        d = torch.sum(d[..., None, :] * pose[:3, :3], -1)
        return pose[None, None, :3, 3].expand(d.shape), d


def test_render_geometry_cast_light_equals_the_reference_method(tmp_path):
    """main.py:634-739 (head close-up, one light draw, Lambert shading of the extra colour, ambience 0) against
    Runner.render_geometry_cast_light under the same numpy seed, fake dataset and fake renderer."""
    import cv2 as cv
    from avatarclip_b200.runner import Runner
    conf = open(os.path.join(HERE, "runner_conf_sample.conf")).read().replace("./exp/CASE_NAME/demo", str(tmp_path / "ours"))
    p = tmp_path / "c.conf"
    p.write_text(conf)
    r = Runner(str(p), mode="validate", case="smpl", device="cpu")
    assert r.head_height == 0.55                                  # the value the reference side was run with
    r.dataset, r.batch_size = CastLightDataset(), 500
    r.renderer.render = FakeRenderer().render
    r.renderer.n_samples, r.renderer.n_importance = 3, 2
    np.random.seed(21)
    path = r.render_geometry_cast_light()
    next_ours = np.random.uniform()
    meta, arrays = _golden()
    ref, ref_img = meta["cast_light"], arrays["cast_light_img"]
    ours = cv.cvtColor(cv.imread(path, cv.IMREAD_UNCHANGED), cv.COLOR_BGR2RGB)
    assert os.path.basename(path) == ref["path"] == "cast_light_texture_head_black.png"
    assert ours.shape == ref_img.shape == (48, 48, 3) and np.array_equal(ours, ref_img)
    assert next_ours == ref["next_uniform"]    # both sides consumed the same draws of numpy's global stream (main.py:671-674)
