"""Runner.train (--mode train, the NeuS pre-fit) against the reference's own loop text (main.py:180-256 + :568-586) on the CPU:
same fake dataset (random pixel batches from torch's global generator), same differentiable fake renderer over the network
parameters, `torch.optim.Adam`, identical seeds.  Pins the loop's host logic -- image permutation cycling, mask handling, the
loss formula, optimiser stepping, WHEN the learning rate is updated, what is logged under which name -- not the renderer (GPU
parity tests).  The reference side was recorded by executing those lines in place on the same fakes
(oracle/pin_host_mirrors.py -> tests/golden/host_mirrors.{json,npz})."""
import json
import os

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden")
CLIP_STEPS = 48
CLIP_CONF_EDITS = (("warm_up_end = 500", "warm_up_end = 5"), ("end_iter = 100000", "end_iter = 80"))


def TRAIN_CONF_EDITS(mask_weight, white):
    return (("end_iter = 100000", "end_iter = 12"), ("warm_up_end = 500", "warm_up_end = 4"), ("batch_size = 512", "batch_size = 40"),
            ("mask_weight = 0.5", f"mask_weight = {mask_weight}"), ("use_white_bkgd = False", f"use_white_bkgd = {white}"),
            ("report_freq = 100", "report_freq = 3"))


def _golden():
    return json.load(open(os.path.join(GOLDEN, "host_mirrors.json")))


class FakeDataset:
    n_images, H, W = 5, 16, 16

    def __init__(self):
        g = torch.Generator().manual_seed(1)
        self.images = torch.rand(5, 16, 16, 3, generator=g)
        self.masks = (torch.rand(5, 16, 16, 1, generator=g) > 0.4).float() * torch.rand(5, 16, 16, 1, generator=g)

    def gen_random_rays_at(self, img_idx, batch_size):
        img_idx = int(img_idx)
        px = torch.randint(low=0, high=self.W, size=[batch_size])
        py = torch.randint(low=0, high=self.H, size=[batch_size])
        d = torch.stack([(px - 8.0) / 16, -(py - 8.0) / 16, -torch.ones(batch_size)], -1)
        d = d / d.norm(dim=-1, keepdim=True)
        o = torch.tensor([0.1 * img_idx, 0.0, 1.5]).expand(batch_size, 3)
        return torch.cat([o, d, self.images[img_idx][(py, px)], self.masks[img_idx][(py, px)]], -1)

    def near_far_from_sphere(self, o, d, is_sphere=False):
        return torch.zeros(o.shape[0], 1), torch.ones(o.shape[0], 1) * 2


def make_render(params):
    def render(rays_o, rays_d, near, far, background_rgb=None, cos_anneal_ratio=0.0, **kw):
        s = sum((p * p).sum() for p in params) * 1e-4 + sum(p.sum() for p in params) * 1e-3
        wsum = torch.sigmoid(rays_o[:, :1] * s + rays_d[:, 1:2] * 3)
        return {"color_fine": torch.sigmoid(rays_d * 2 + s), "s_val": wsum * 0.1 + s, "cdf_fine": wsum.expand(-1, 4) * 0.5,
                "gradient_error": (s - 0.3) ** 2, "weight_max": wsum * 0.5, "weight_sum": wsum, "extra_color_fine": None}
    return render


class Writer:
    def __init__(self):
        self.rec = []

    def add_scalar(self, name, value, step):
        self.rec.append((name, float(value), int(step)))


@pytest.mark.parametrize("mask_weight,white", [(0.5, False), (0.0, True)])
def test_mode_train_loop_equals_the_reference_loop(tmp_path, mask_weight, white):
    from avatarclip_b200.runner import Runner
    conf = open(os.path.join(HERE, "runner_conf_sample.conf")).read().replace("./exp/CASE_NAME/demo", str(tmp_path / "ours"))
    for old, new in TRAIN_CONF_EDITS(mask_weight, white):
        assert old in conf
        conf = conf.replace(old, new)
    p = tmp_path / "c.conf"
    p.write_text(conf)
    r = Runner(str(p), mode="train", case="smpl", device="cpu")
    r.dataset = FakeDataset()
    key = f"{mask_weight}_{white}"
    ref = _golden()["train_loop"][key]
    arrays = np.load(os.path.join(GOLDEN, "host_mirrors.npz"))
    wr = Writer()
    r._make_writer = lambda: wr
    r.save_freq = r.val_freq = r.val_mesh_freq = 10 ** 9
    r.renderer.render = make_render(r._all_params())
    torch.manual_seed(7)
    logs = []
    assert r.train(log=logs.append, validate=False) == 12 == ref["iter_step"]
    assert [n for n, _, _ in wr.rec] == [n for n, _, _ in ref["rec"]]                # same scalar names in the same order
    assert [s for _, _, s in wr.rec] == [s for _, _, s in ref["rec"]]
    worst = max(abs(a - b) / max(abs(b), 1e-12) for (_, a, _), (_, b, _) in zip(wr.rec, ref["rec"]))
    assert worst < 1e-6, worst
    params = list(r._all_params())                                                   # the same parameters after 12 Adam steps
    assert len(params) == ref["n_params"] and [list(q.shape) for q in params] == ref["param_shapes"]
    for i, a in enumerate(params):                                                   # on a fixed, seeded sample of each tensor
        idx = torch.from_numpy(arrays[f"train_loop_{key}_param{i}_idx"]).long()
        want = torch.from_numpy(arrays[f"train_loop_{key}_param{i}_val"])
        assert torch.allclose(a.detach().reshape(-1)[idx], want, rtol=1e-6, atol=1e-9), i
    assert r.optimizer.param_groups[0]["lr"] == ref["final_lr"]
    lr_ours = [str(m).split("lr=")[1] for m in logs if "lr=" in str(m)]
    assert lr_ours == ref["lr_printed"] and len(lr_ours) == 4                        # the lr in force at steps 3, 6, 9, 12


def test_train_clip_host_logic_equals_the_reference_lines(tmp_path, monkeypatch):
    """What Runner.train_clip hands to the fused step, step by step -- camera pose, background mode, light, ambience (numpy's
    global stream seeded by train.seed), WHICH cached text embedding (main.py:499-507: face every 4th step, back when the camera
    is behind, else body), the learning rate in force (update_learning_rate before the loop and after every step, :339,563)
    and the cosine-anneal ratio -- against what the reference's own lines gave for the same seed and conf.  The step itself is
    mocked (GPU tests)."""
    import types
    from avatarclip_b200 import views
    from avatarclip_b200.runner import Runner
    conf = open(os.path.join(HERE, "runner_conf_sample.conf")).read().replace("./exp/CASE_NAME/demo", str(tmp_path / "ours"))
    for old, new in CLIP_CONF_EDITS:
        conf = conf.replace(old, new)
    p = tmp_path / "c.conf"
    p.write_text(conf)
    r = Runner(str(p), mode="train_clip", case="smpl", device="cpu")                  # seeds numpy with train.seed = 11
    body, face, back = torch.zeros(1, 4), torch.ones(1, 4), torch.full((1, 4), 2.0)
    r.encoded_text, r.encoded_face_text, r.encoded_back_text = body, face, back
    r.clip_tower, r.v, r.f = object(), torch.zeros(1, 3, 3), np.zeros((1, 3), dtype=np.int64)
    r.dataset = types.SimpleNamespace(H=256, W=256, focal=221.7, n_images=0)
    rec = []

    class FakeTrainer:
        iter_step, scalars, cos, _out = 0, None, None, None

        def set_text(self, emb):
            self.text = emb

        def step(self, view, lr=None, cos_anneal=1.0):
            d = view.draw
            rec.append(dict(text=float(self.text[0, 0]), lr=lr, cos_anneal=cos_anneal, pose=d.pose.copy(), bg=d.bg_choice,
                            light=d.light_dir.copy(), ambience=d.ambience, face=d.face_step, is_front=d.is_front))
            return torch.tensor(1.0)

    class FakeBuilder:
        def __init__(self, *a, **k):
            pass

        def submit(self, draw):
            return draw

        def finish(self, pending):
            return types.SimpleNamespace(draw=pending)

    r.trainer = FakeTrainer()
    monkeypatch.setattr(views, "ViewBuilder", FakeBuilder)
    r._make_writer = lambda: __import__("avatarclip_b200.runner", fromlist=["_NullWriter"])._NullWriter()
    assert r.train_clip(max_steps=CLIP_STEPS, log=lambda m: None, validate=False) == CLIP_STEPS
    ref = _golden()["train_clip"]
    assert len(ref) == len(rec) == CLIP_STEPS
    for i, (got, want) in enumerate(zip(rec, ref)):
        assert got["text"] == want["text"] == want["no_texture_text"], i
        assert got["lr"] == want["lr"], i
        assert got["cos_anneal"] == want["cos_anneal"]
        assert np.array_equal(got["pose"], np.asarray(want["pose"])) and got["bg"] == want["bg"], i
        assert np.array_equal(got["light"], np.asarray(want["light"], dtype=np.float32)) and got["ambience"] == want["ambience"]
    assert {g["text"] for g in rec} == {0.0, 1.0, 2.0}             # body, face and back prompts all occurred
