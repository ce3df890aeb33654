"""Runner mirror: conf-driven construction, LR schedule, checkpoint layout (CPU); the real train_clip loop (per-step
draws, device view preparation with lookahead, prompt selection, resume in the CLI order), --mode train on a hand-off
directory, validation image / mesh outputs (GPU)."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import loss as ol

HERE = os.path.dirname(os.path.abspath(__file__))
CONF = os.path.join(HERE, "runner_conf_sample.conf")
GOLDEN = os.path.join(HERE, "golden")


def _conf_text(tmp_path, data_dir=None, edits=()):
    text = open(CONF).read().replace("./exp/CASE_NAME/demo", str(tmp_path / "exp"))
    for old, new in edits:
        assert old in text
        text = text.replace(old, new)
    if data_dir is not None:
        text = text.replace("./data/zero_beta_tpose_render", str(data_dir))
    p = tmp_path / "run.conf"
    p.write_text(text)
    return str(p)


def _runner(tmp_path, device, mode="train_clip", data_dir=None, is_continue=False, edits=()):
    from avatarclip_b200.runner import Runner
    return Runner(_conf_text(tmp_path, data_dir, edits), mode=mode, case="smpl", device=device, is_continue=is_continue)


def test_runner_construction_schedule_and_checkpoint_layout(tmp_path):
    r = _runner(tmp_path, "cpu", mode="validate")
    assert r.use_face_prompt and r.use_back_prompt and r.head_height == 0.55 and r.seed == 11
    for it in (0, 100, 499, 500, 5000, 99999):
        r.iter_step = it
        want = 5e-4 * ol.learning_rate_factor(it, 500.0, 100000, 0.05)
        assert abs(r.current_lr() - want) < 1e-12
    assert r.get_cos_anneal_ratio() == 1.0
    r.iter_step = 7
    path = r.save_checkpoint()
    ck = torch.load(path, weights_only=False)
    assert set(ck.keys()) == {"sdf_network_fine", "variance_network_fine", "color_network_fine", "optimizer", "iter_step"}
    assert list(ck["sdf_network_fine"].keys())[:3] == ["lin0.bias", "lin0.weight_g", "lin0.weight_v"]
    assert ck["iter_step"] == 7 and os.path.basename(path) == "ckpt_000007.pth"
    # the reference's optimizer (main.py:141-145) accepts the stored optimizer state
    params = list(r.sdf_network.parameters()) + list(r.deviation_network.parameters()) + list(r.color_network.parameters())
    torch.optim.Adam(params, lr=5e-4).load_state_dict(ck["optimizer"])
    r2 = _runner(tmp_path, "cpu", mode="validate")
    r2.load_checkpoint(path)
    assert r2.iter_step == 7
    for a, b in zip(r.sdf_network.parameters(), r2.sdf_network.parameters()):
        assert torch.equal(a, b)


def test_cli_dispatch_mirrors_the_reference_main(monkeypatch):
    """main.py:953-979: flags, `is_continue` forced for the two inference modes, and what each mode calls, in order."""
    from avatarclip_b200 import runner as R
    calls = []

    class Fake:
        def __init__(self, conf, mode, case, is_continue, device=None):
            calls.append(("init", conf, mode, case, is_continue, device))

        def __getattr__(self, name):
            return lambda *a, **k: calls.append((name, a, k))

    monkeypatch.setattr(R, "Runner", Fake)
    monkeypatch.setattr(R.torch.cuda, "set_device", lambda i: calls.append(("set_device", i)))
    R.main(["--conf", "c.conf", "--mode", "validate_mesh", "--case", "x", "--gpu", "0", "--mcube_threshold", "0.25"])
    assert calls[0] == ("set_device", 0) and calls[1] == ("init", "c.conf", "validate_mesh", "x", True, "cuda:0")
    assert calls[2] == ("validate_mesh", (), {"world_space": True, "resolution": 512, "threshold": 0.25})
    assert calls[3][0] == "render_geometry_cast_light" and len(calls) == 4
    calls.clear()
    R.main(["--conf", "c.conf", "--mode", "train_clip"])
    assert calls[1] == ("init", "c.conf", "train_clip", "smpl", False, "cuda:0")
    assert [c[0] for c in calls[2:]] == ["init_clip", "init_smpl", "train_clip"]
    calls.clear()
    R.main(["--conf", "c.conf", "--mode", "render_geometry_cast_light"])
    assert calls[1][4] is True and [c[0] for c in calls[2:]] == ["render_geometry_cast_light"]
    calls.clear()
    R.main(["--conf", "c.conf", "--mode", "train", "--is_continue"])
    assert calls[1][2] == "train" and calls[1][4] is True and [c[0] for c in calls[2:]] == ["train"]
    with pytest.raises(SystemExit):
        R.main(["--conf", "c.conf", "--mode", "nonsense"])


def _clip_args():
    from avatarclip_b200.workload import random_vit_state
    g = torch.Generator().manual_seed(0)
    return random_vit_state(seed=0), torch.randn(1, 512, generator=g), torch.randn(1, 512, generator=g), \
        torch.randn(1, 512, generator=g)


@pytest.mark.gpu
def test_runner_train_clip_real_loop_and_cli_order_resume(tmp_path):
    """train_clip with NO view_source: cameras from the seeded sampler, template rasterised and silhouette rays prepared
    on the device one step ahead, face / back prompts selected per step; then resume like the CLI does
    (Runner(is_continue=True) BEFORE init_clip -- ADVICE r1: the Adam moments must survive)."""
    from avatarclip_b200.workload import synthetic_body_mesh
    sd, text, face, back = _clip_args()
    v, f = synthetic_body_mesh(12, 16)
    r = _runner(tmp_path, "cuda")
    r.init_clip(sd, text, face, back)
    r.init_smpl(v, f)
    used = []
    orig = r._ensure_trainer().set_text
    r.trainer.set_text = lambda e: (used.append(e.data_ptr()), orig(e))[1]
    logs = []
    before = r.sdf_network.lin1.weight_v.detach().clone()
    r.report_freq = 2
    assert r.train_clip(max_steps=6, log=logs.append, validate=False) == 6
    assert not torch.equal(before, r.sdf_network.lin1.weight_v)
    assert any("loss" in str(l) for l in logs)
    assert used[0] == r.encoded_face_text.data_ptr() and used[4] == r.encoded_face_text.data_ptr()   # iter_i % 4 == 0
    assert all(u in (r.encoded_text.data_ptr(), r.encoded_back_text.data_ptr()) for i, u in enumerate(used) if i % 4)
    # a ray count above the renderer's chunk (4096) and different every step: chunked forward + recompute backward, output
    # buffers re-sized per step
    r.max_ray_num = 5000
    r.report_freq = 1
    logs2, rays = [], []
    for _ in range(2):
        assert r.train_clip(max_steps=2, log=logs2.append, validate=False) == r.iter_step      # a face step + a body step
        rays.append(int(r.trainer._out["weights"].shape[0]))
    vals = [float(str(m).split("loss = ")[1].split(" ")[0]) for m in logs2 if "loss = " in str(m)]
    assert len(vals) == 4 and all(np.isfinite(vals)) and max(rays) > 4096 and max(rays) < 5200, (vals, rays)
    r.max_ray_num = 600
    path = r.save_checkpoint()
    ck = torch.load(path, weights_only=False)
    assert len(ck["optimizer"]["state"]) == len(r._all_params())
    torch.optim.Adam(r._all_params(), lr=5e-4).load_state_dict(ck["optimizer"])       # reference-format Adam state
    # CLI order: constructor (loads the checkpoint) first, init_clip afterwards
    r2 = _runner(tmp_path, "cuda", is_continue=True)
    assert r2.iter_step == 10 and r2.trainer is None and r2._pending_optimizer_state is not None
    r2.init_clip(sd, text, face, back)
    tr2 = r2._ensure_trainer()
    assert tr2.iter_step == 10 and torch.equal(tr2.exp_avg, r.trainer.exp_avg) and torch.equal(tr2.exp_avg_sq, r.trainer.exp_avg_sq)
    assert float(tr2.exp_avg.abs().max()) > 0
    img = r2.render_image(ol.lookat([0.0, 0.0, 1.6], [0.0, 0.0, 0.0]), resolution_level=8)
    assert img.shape == (32, 32, 3) and torch.isfinite(img).all()


# the switch settings of confs/ablation/*_0.conf, *_1.conf, *_2.conf (no face / back prompts there)
_NO_PROMPTS = (("use_face_prompt = True", "use_face_prompt = False"), ("use_back_prompt = True", "use_back_prompt = False"))
ABLATIONS = {
    "0": _NO_PROMPTS + (("add_no_texture = True", "add_no_texture = False"), ("texture_cast_light = True", "texture_cast_light = False"),
                        ("use_silhouettes = True", "use_silhouettes = True\n    use_bg_aug = False")),
    "1": _NO_PROMPTS + (("add_no_texture = True", "add_no_texture = False"), ("texture_cast_light = True", "texture_cast_light = False")),
    "2": _NO_PROMPTS + (("texture_cast_light = True", "texture_cast_light = False"),),
}


def test_ablation_confs_construct_with_their_switches(tmp_path):
    r = _runner(tmp_path, "cpu", mode="validate", edits=ABLATIONS["0"])
    assert not (r.add_no_texture or r.texture_cast_light or r.use_bg_aug or r.use_face_prompt or r.use_back_prompt)
    r = _runner(tmp_path, "cpu", mode="validate", edits=ABLATIONS["2"])
    assert r.add_no_texture and not r.texture_cast_light and r.use_bg_aug


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["0", "1", "2"])
def test_runner_train_clip_with_the_ablation_conf_switches(tmp_path, variant):
    """The 18 confs under confs/ablation/*_{0,1,2}.conf switch add_no_texture / texture_cast_light (and use_bg_aug) off
    (main.py:388-391,425,509-534): the real loop runs them -- finite losses, parameters move, the loss of a
    step without the shading term is the base loss plus ONE CLIP term."""
    from avatarclip_b200.workload import synthetic_body_mesh
    from avatarclip_b200 import losses as PL
    sd, text, _, _ = _clip_args()
    v, f = synthetic_body_mesh(12, 16)
    r = _runner(tmp_path, "cuda", edits=ABLATIONS[variant])
    r.init_clip(sd, text)
    r.init_smpl(v, f)
    r.report_freq = 1
    logs = []
    before = r.color_network.lin0.weight_v.detach().clone()
    assert r.train_clip(max_steps=3, log=logs.append, validate=False) == 3
    vals = [float(str(m).split("loss = ")[1].split(" ")[0]) for m in logs if "loss = " in str(m)]
    assert len(vals) == 3 and all(np.isfinite(vals))
    assert not torch.equal(before, r.color_network.lin0.weight_v)
    tr = r.trainer
    n_terms = 2 if r.add_no_texture else 1
    want = tr.scalars[PL.S_BASE] + ((1.0 - tr.cos[:n_terms]) * tr.clip_weight).sum()
    assert abs(float(tr.loss_value()) - float(want)) < 1e-6
    assert (tr.add_no_texture, tr.texture_cast_light) == (r.add_no_texture, r.texture_cast_light)


@pytest.mark.gpu
@pytest.mark.parametrize("extra_color", [True, False])
def test_mode_train_on_handoff_directory_and_validation_outputs(tmp_path, extra_color):
    """ShapeGen hand-off (108 rendered views + transforms_train.json) -> SMPL_Dataset -> --mode train (NeuS pre-fit
    through the autograd seam + torch.optim.Adam) -> validate_image PNGs and validate_mesh PLY.  extra_color False is the
    network of confs/base_models/astrongman.conf (the conf --mode train ships with): no second colour head, the fixed
    background blends into `color` (models/renderer.py:272-281)."""
    edits = () if extra_color else (("        extra_color = True\n", ""),)
    from avatarclip_b200.handoff import read_ply, render_coarse_shape
    from avatarclip_b200.workload import synthetic_body_mesh
    v, f = synthetic_body_mesh(12, 16)
    data_dir = tmp_path / "render"
    render_coarse_shape(v, f, str(data_dir), image_size=64)
    meta = json.load(open(data_dir / "transforms_train.json"))
    assert len(meta["frames"]) == 108 and abs(meta["camera_angle_x"] - np.pi / 3) < 1e-12
    r = _runner(tmp_path, "cuda", mode="train", data_dir=data_dir, edits=edits)
    assert r.dataset.n_images == 108 and r.dataset.H == 64 and float(r.dataset.masks.mean()) > 0.01
    assert r.extra_color == extra_color == r.renderer.extra_color == hasattr(r.color_network, "extra_lin")
    r.batch_size = 256
    # the training loss of main.py:204-224 on a FIXED batch with a FIXED jitter draw (the logged per-step values belong to a
    # different random image / pixel batch every step and the learning rate is still in its warm-up: noise, not descent)
    import torch.nn.functional as F
    data = r.dataset.gen_random_rays_at(5, 256)
    jit = torch.rand(256, device="cuda") - 0.5

    def fixed_batch_loss():
        with torch.no_grad():
            ro, rd, true_rgb, mask = data[:, :3], data[:, 3:6], data[:, 6:9], (data[:, 9:10] > 0.5).float()
            near, far = r.dataset.near_far_from_sphere(ro, rd)
            out = r.renderer.render(ro, rd, near, far, jitter=jit, cos_anneal_ratio=r.get_cos_anneal_ratio())
            color = ((out["color_fine"] - true_rgb) * mask).abs().sum() / (mask.sum() + 1e-5)
            bce = F.binary_cross_entropy(out["weight_sum"].clip(1e-3, 1.0 - 1e-3), mask)
            return float(color + out["gradient_error"] * r.igr_weight + bce * r.mask_weight)

    before_w = r.sdf_network.lin1.weight_v.detach().clone()
    loss_before = fixed_batch_loss()
    losses = []
    r.report_freq = 5
    r.train(max_steps=30, log=lambda m: losses.append(m), validate=False)
    loss_after = fixed_batch_loss()
    vals = [float(str(m).split("loss = ")[1].split(" ")[0]) for m in losses if "loss = " in str(m)]
    print(f"extra_color {extra_color}: fixed-batch loss {loss_before:.5f} -> {loss_after:.5f}; logged {vals}")
    assert len(vals) == 6 and all(np.isfinite(vals)) and np.isfinite(loss_before) and np.isfinite(loss_after)
    assert not torch.equal(before_w, r.sdf_network.lin1.weight_v)
    assert loss_after < loss_before
    img, extra, normal = r.validate_image(idx=3, resolution_level=2)
    assert img.shape == (32, 32, 3) and (extra is None) == (not extra_color)
    if not extra_color:
        # renderer.py:277-281 without the extra head: color = color + background * (1 - weight_sum), differentiable
        ro, rd = r.dataset.gen_rays_at(3, resolution_level=4)
        ro, rd = ro.reshape(-1, 3)[:200], rd.reshape(-1, 3)[:200]
        near, far = r.dataset.near_far_from_sphere(ro, rd)
        jit = torch.rand(200, device="cuda") - 0.5
        plain = r.renderer.render(ro, rd, near, far, jitter=jit, cos_anneal_ratio=1.0)
        white = r.renderer.render(ro, rd, near, far, jitter=jit, cos_anneal_ratio=1.0,
                                  background_rgb=torch.ones([1, 3], device="cuda"))
        assert plain["extra_color_fine"] is None and white["extra_color_fine"] is None
        assert torch.allclose(white["color_fine"], plain["color_fine"] + (1.0 - plain["weight_sum"]), atol=1e-6)
        for p in r._all_params():
            p.grad = None
        white["color_fine"].sum().backward()
        assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in r._all_params())
        assert "extra_lin.bias" not in r.color_network.state_dict()
    assert os.path.exists(os.path.join(r.base_exp_dir, "validations_fine", "{:0>8d}_0_3.png".format(r.iter_step)))
    assert os.path.exists(os.path.join(r.base_exp_dir, "normals", "{:0>8d}_0_3.png".format(r.iter_step)))
    path = r.validate_mesh(resolution=48)
    vv, ff, cc = read_ply(path)
    assert vv.shape[0] > 100 and ff.shape[0] > 100 and cc.shape == (vv.shape[0], 3)
    assert ff.max() < vv.shape[0] and np.abs(vv).max() <= 1.02
    # resume --mode train with the torch optimizer state
    ck = r.save_checkpoint()
    r2 = _runner(tmp_path, "cuda", mode="train", data_dir=data_dir, is_continue=True, edits=edits)
    opt = r2._ensure_optimizer()
    assert r2.iter_step == 30 and len(opt.state) == len(r2._all_params())


@pytest.mark.gpu
def test_extract_geometry_sphere_is_watertight_and_outward(tmp_path):
    """Marching tetrahedra on the geometric-init SDF (a sphere of radius ~0.5): vertices on the iso-surface, every edge
    shared by exactly two triangles, normals pointing out of the body; boundary evaluators against the oracle."""
    import util_neus as U
    from oracle import neus
    sdf_kw, col_kw, ren_kw, _ = U.CASES["b2"]            # untamed geometric init of the 8x256 net: |x| - 0.5, smooth
    sconf, _, _ = U.confs_from_kw(sdf_kw, col_kw, ren_kw)
    sp, cp = U.synth_state(sdf_kw, col_kw, 3, tame=False)
    sdf, col, var, ren = U.build_product(sdf_kw, col_kw, ren_kw, sp, cp, 0.3, "cuda", engine=1)
    verts, tris = ren.extract_geometry([-1.01] * 3, [1.01] * 3, resolution=64, threshold=0.0)
    assert verts.shape[0] > 500 and tris.shape[0] > 1000
    s = neus.sdf_value(sp, sconf, torch.from_numpy(verts).float()).reshape(-1)
    assert float(s.abs().max()) < 2e-3      # linear interpolation on a 64^3 grid (measured on the CPU field: 1.1e-3)
    assert abs(float(np.linalg.norm(verts, axis=1).mean()) - 0.5) < 0.01
    e = np.concatenate([tris[:, [0, 1]], tris[:, [1, 2]], tris[:, [2, 0]]])
    key = np.sort(e, axis=1)
    _, counts = np.unique(key[:, 0].astype(np.int64) * verts.shape[0] + key[:, 1], return_counts=True)
    assert (counts == 2).all()
    a, b, c = verts[tris[:, 0]], verts[tris[:, 1]], verts[tris[:, 2]]
    n = np.cross(b - a, c - a)
    assert ((n * (a + b + c)).sum(1) > 0).mean() > 0.999    # outward on a sphere centred at the origin
    # SDFNetwork.forward / gradient (models/fields.py:72-107) against the oracle's autograd
    pts = ((torch.rand(3000, 3) - 0.5) * 1.6)
    out = sdf(pts.cuda()).cpu()
    want = neus.sdf_forward(sp, sconf, pts)              # [P, d_out] = (sdf, features)
    assert out.shape == (3000, sdf_kw["d_out"]) and U.rel_to_max(out, want) < 1e-5
    assert U.rel_to_max(out[:, :1], neus.sdf_value(sp, sconf, pts)) < 1e-5
    g = sdf.gradient(pts.cuda()).cpu()
    p = pts.clone().requires_grad_(True)
    (gw,) = torch.autograd.grad(neus.sdf_value(sp, sconf, p).sum(), p)
    assert g.shape == (3000, 1, 3) and U.rel_to_max(g[:, 0], gw) < 1e-4
    assert torch.equal(sdf.sdf_hidden_appearance(pts.cuda()).cpu(), out)


def _shipped_checkpoint(path):
    """pretrained_models/zero_beta_stand_pose.pth's three network state dicts, rebuilt from the tensors tests/golden/neus_shipped.pt
    carries, in the file's key order, each tensor checked against the sha256 recorded from the shipped file
    (oracle/pin_host_mirrors.py)."""
    import hashlib
    g = torch.load(os.path.join(GOLDEN, "neus_shipped.pt"), weights_only=False)
    ref = json.load(open(os.path.join(GOLDEN, "host_mirrors.json")))["checkpoint"]
    src = {"sdf_network_fine": g["sdf_state"], "color_network_fine": g["col_state"], "variance_network_fine": {"variance": g["variance"]}}
    ck = {}
    for part, want in ref.items():
        ck[part] = {k: src[part][k].clone() for k in want["keys"]}
        for (k, v), h in zip(ck[part].items(), want["sha256"]):
            assert hashlib.sha256(np.ascontiguousarray(v.numpy()).tobytes()).hexdigest() == h, (part, k)
    torch.save(ck, path)
    return ck


def test_shipped_example_conf_constructs_a_runner_and_loads_the_shipped_checkpoint(tmp_path):
    """confs/examples/ironman.conf as shipped (only the three relative paths made absolute, because the test does not run from
    inside the reference tree): the Runner builds the networks from the conf subtrees, reads every train.* key and loads
    `train.pretrain` = pretrained_models/zero_beta_stand_pose.pth like main.py:153-160,612-619."""
    import tarfile
    from avatarclip_b200.runner import Runner
    with tarfile.open(os.path.join(GOLDEN, "shipped_confs.tar.xz")) as tf:
        text = tf.extractfile("confs/examples/ironman.conf").read().decode()
    (tmp_path / "pretrained_models").mkdir()
    ck = _shipped_checkpoint(str(tmp_path / "pretrained_models" / "zero_beta_stand_pose.pth"))
    for old, new in (("./exp/", str(tmp_path / "exp") + "/"), ("./data/", str(tmp_path / "data") + "/"),
                     ("./pretrained_models/", str(tmp_path / "pretrained_models") + "/")):
        assert old in text
        text = text.replace(old, new)
    p = tmp_path / "ironman.conf"
    p.write_text(text)
    r = Runner(str(p), mode="validate", case="smpl", device="cpu")
    assert (r.use_silhouettes, r.add_no_texture, r.texture_cast_light, r.use_face_prompt, r.use_back_prompt, r.extra_color) == (True,) * 6
    assert r.max_ray_num == 112 * 112 and r.end_iter == 100000 and r.renderer.n_samples == 32 and r.renderer.n_importance == 32
    for k, v in ck["sdf_network_fine"].items():
        assert torch.equal(r.sdf_network.state_dict()[k], v), k
    assert torch.equal(r.deviation_network.variance.detach(), ck["variance_network_fine"]["variance"])
    for k, v in ck["color_network_fine"].items():                     # the file has no extra_lin (main.py:617 strict=False)
        assert torch.equal(r.color_network.state_dict()[k], v), k
    assert "extra_lin.weight_v" in r.color_network.state_dict() and "extra_lin.weight_v" not in ck["color_network_fine"]
    assert abs(r.current_lr()) == 0.0 and r.get_cos_anneal_ratio() == 1.0          # iter 0 of the warm-up; anneal_end = 0
