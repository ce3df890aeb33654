"""Records what the host-side mirror tests compare against, by running the UNMODIFIED reference's own code and data once:

    python -m oracle.pin_host_mirrors          # needs the reference checkout (oracle.pin_loss_stage.REF)

Writes, under tests/golden/:
  shipped_confs.tar.xz         the reference's confs/ tree (180 .conf files, data fixtures)
  shipped_render_sample/       4 of the 108 frames of each shipped render directory (PNGs + trimmed transforms_train.json)
  zero_beta_smpl_sample.obj    the first 700 vertices of the shipped SMPL template and the faces among them, lines verbatim
  host_mirrors.json / .npz     the reference side of tests/test_{fields,dataset,handoff,runner,train_loop,validate}_cpu.py:
                               constructor states (sha256 per tensor), the dataset constructor's tensors on the sample
                               directories, ShapeGen's camera matrices, the shipped checkpoint's key order and hashes,
                               the --mode train loop's logged scalars / lr / parameters, train_clip's per-step schedule,
                               and the files validate_image / validate_mesh / render_geometry_cast_light write.
The tests replay these without the reference checkout; the fake datasets / renderers both sides run on are the tests' own.
"""
from __future__ import annotations

import contextlib
import copy
import hashlib
import io
import json
import os
import shutil
import sys
import tarfile
import types

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
GOLDEN = os.path.join(ROOT, "tests", "golden")

from oracle import make_ref                      # noqa: E402
from oracle.pin_loss_stage import REF, cut       # noqa: E402

SAMPLE_FRAMES = (0, 29, 58, 107)
OBJ_SAMPLE_VERTS = 700


def tensor_sha(t) -> str:
    a = np.ascontiguousarray(t.detach().cpu().numpy() if torch.is_tensor(t) else np.asarray(t))
    return hashlib.sha256(a.tobytes()).hexdigest()


def state_digest(module) -> dict:
    sd = module.state_dict()
    return {"keys": list(sd.keys()), "shapes": [list(v.shape) for v in sd.values()], "sha256": [tensor_sha(v) for v in sd.values()],
            "param_names": [n for n, _ in module.named_parameters()]}


def param_sample(t, n=256, seed=0):
    """A fixed, seeded sample of a tensor's entries (flat indices, values)."""
    flat = t.detach().reshape(-1)
    idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(seed))[:n].sort().values
    return idx.numpy().astype(np.int32), flat[idx].numpy()


# ---------------------------------------------------------------------------------------------------- tests/test_conf_cpu.py
def pin_confs():
    with tarfile.open(os.path.join(GOLDEN, "shipped_confs.tar.xz"), "w:xz", preset=9) as tf:
        for d, _, files in sorted(os.walk(os.path.join(REF, "confs"))):
            for name in sorted(f for f in files if f.endswith(".conf")):
                full = os.path.join(d, name)
                info = tf.gettarinfo(full, arcname=os.path.relpath(full, REF))
                info.uid = info.gid = 0
                info.uname = info.gname = ""
                info.mtime = 0
                info.mode = 0o644
                with open(full, "rb") as f:
                    tf.addfile(info, f)


# -------------------------------------------------------------------------------------------------- tests/test_fields_cpu.py
def pin_fields():
    import test_fields_cpu as T
    fields, _ = make_ref.load_reference_models()
    out = {}
    for name, kw, cls, seed in (("sdf_shipped", T.SDF_S, fields.SDFNetwork, 0), ("sdf_b2", T.SDF_B2, fields.SDFNetwork, 0),
                                ("sdf_small", T.SDF_SMALL, fields.SDFNetwork, 0),
                                ("col_extra", dict(T.COL, extra_color=True), fields.RenderingNetwork, 3),
                                ("col_plain", dict(T.COL, extra_color=False), fields.RenderingNetwork, 3)):
        torch.manual_seed(seed)
        m = cls(**kw)
        out[name] = dict(state_digest(m), rand_after=float(torch.rand(1)), has_extra_lin=hasattr(m, "extra_lin"))
    out["variance"] = state_digest(fields.SingleVarianceNetwork(0.3))
    return out


# ------------------------------------------------------------------------------------------------- tests/test_dataset_cpu.py
def _reference_dataset(data_dir):
    import cv2 as cv

    class _Conf(dict):
        def get_string(self, k):
            return self[k]

    body = cut("models/dataset.py", 204, 250, "def __init__(self, conf)", "Load data: End")
    body = body.replace("torch.device('cuda')", "torch.device('cpu')").replace("super(SMPL_Dataset, self).__init__()", "pass")

    def imread(fname):
        img = cv.imread(fname, cv.IMREAD_UNCHANGED)
        return img[:, :, [2, 1, 0] + ([3] if img.shape[2] == 4 else [])]

    ns = dict(np=np, torch=torch, os=os, json=json, imageio=type("I", (), {"imread": staticmethod(imread)}),
              pose_spherical=lambda *a: torch.eye(4))
    exec(body, ns)
    obj = type("RefDataset", (), {})()
    ns["__init__"](obj, _Conf(data_dir=data_dir))
    return obj


def pin_dataset():
    out = {}
    for name in ("zero_beta_tpose_render", "zero_beta_standpose_render"):
        src = os.path.join(REF, "data", name)
        dst = os.path.join(GOLDEN, "shipped_render_sample", name)
        shutil.rmtree(dst, ignore_errors=True)
        os.makedirs(os.path.join(dst, "img"))
        meta = json.load(open(os.path.join(src, "transforms_train.json")))
        assert len(meta["frames"]) == 108
        meta["frames"] = [meta["frames"][i] for i in SAMPLE_FRAMES]
        for fr in meta["frames"]:
            shutil.copyfile(os.path.join(src, fr["file_path"] + ".png"), os.path.join(dst, fr["file_path"] + ".png"))
        with open(os.path.join(dst, "transforms_train.json"), "w") as f:
            json.dump(meta, f, indent=1)
        ref = _reference_dataset(dst)
        out[name] = {"n_images": ref.n_images, "H": int(ref.H), "W": int(ref.W), "focal": float(ref.focal),
                     "image_pixels": int(ref.image_pixels),
                     "images": tensor_sha(ref.images), "masks": tensor_sha(ref.masks), "poses": tensor_sha(ref.poses),
                     "K": tensor_sha(ref.K), "shapes": {k: list(getattr(ref, k).shape) for k in ("images", "masks", "poses", "K")},
                     "object_bbox_min": ref.object_bbox_min.tolist(), "object_bbox_max": ref.object_bbox_max.tolist(),
                     "images_lis": [os.path.relpath(p, dst) for p in ref.images_lis]}
    return out


# ------------------------------------------------------------------------------------------------- tests/test_handoff_cpu.py
def pin_handoff(arrays):
    from avatarclip_b200 import handoff
    ns = {"np": np}
    exec(cut("../ShapeGen/render.py", 16, 30, "def norm_np_arr", "return viewMatrix"), ns)
    mats = []
    for a in range(0, 360, 40):
        for e in (-60, -20, 0, 40):
            eye = handoff.get_points_from_angles(2.2, e, a)
            mats.append(ns["lookat"](eye, np.array([0, 0, 0]), np.array([0, 1, 0]))[0])
    arrays["handoff_lookat"] = np.stack(mats).astype(np.float64)
    # the template sample: its first OBJ_SAMPLE_VERTS vertex lines and the face lines among them, verbatim and in order
    lines = open(os.path.join(REF, "data", "zero_beta_smpl.obj")).read().split("\n")
    vl = [l for l in lines if l.startswith("v ")]
    fl = [l for l in lines if l.startswith("f ")]
    assert len(vl) == 6890 and len(fl) == 13776 and all(l.startswith(("v ", "f ")) or not l.strip() for l in lines)
    keep_f = [l for l in fl if max(int(t.split("/")[0]) for t in l.split()[1:]) <= OBJ_SAMPLE_VERTS]
    with open(os.path.join(GOLDEN, "zero_beta_smpl_sample.obj"), "w") as f:
        f.write("\n".join(vl[:OBJ_SAMPLE_VERTS] + keep_f) + "\n")
    fi = np.array([[int(t) - 1 for t in l.split()[1:]] for l in keep_f])
    return {"obj_sample": {"n_verts": OBJ_SAMPLE_VERTS, "n_faces": len(keep_f), "face_min": int(fi.min()), "face_max": int(fi.max()),
                           "full_template": {"n_verts": len(vl), "n_faces": len(fl)}}}


# ------------------------------------------------------------------------------------------------------ tests/test_runner.py
def pin_checkpoint():
    ck = torch.load(os.path.join(REF, "pretrained_models", "zero_beta_stand_pose.pth"), map_location="cpu", weights_only=False)
    return {part: {"keys": list(ck[part].keys()), "sha256": [tensor_sha(v) for v in ck[part].values()]}
            for part in ("sdf_network_fine", "variance_network_fine", "color_network_fine")}


# ---------------------------------------------------------------------------------------------- tests/test_train_loop_cpu.py
def _train_loop_case(tmp, mask_weight, white, arrays, key):
    import test_train_loop_cpu as T
    from avatarclip_b200.runner import Runner
    os.makedirs(tmp)
    conf = open(os.path.join(ROOT, "tests", "runner_conf_sample.conf")).read().replace("./exp/CASE_NAME/demo", os.path.join(tmp, "ours"))
    for old, new in T.TRAIN_CONF_EDITS(mask_weight, white):
        conf = conf.replace(old, new)
    p = os.path.join(tmp, "c.conf")
    open(p, "w").write(conf)
    r = Runner(p, mode="train", case="smpl", device="cpu")
    nets = [copy.deepcopy(m) for m in (r.sdf_network, r.deviation_network, r.color_network)]
    ref_params = [q for m in nets for q in m.parameters()]
    ns = dict(np=np, torch=torch, F=F, os=os, tqdm=lambda it: it)
    exec(cut("main.py", 180, 256, "def train(self):", "image_perm = self.get_image_perm()"), ns)
    exec(cut("main.py", 568, 586, "def get_image_perm(self):", "g['lr']"), ns)
    wr_ref = T.Writer()
    ns["SummaryWriter"] = lambda log_dir=None: wr_ref
    ref = types.SimpleNamespace(
        base_exp_dir=os.path.join(tmp, "ref"), end_iter=12, iter_step=0, dataset=T.FakeDataset(), batch_size=40, use_white_bkgd=white,
        mask_weight=mask_weight, igr_weight=r.igr_weight, report_freq=3, save_freq=10 ** 9, val_freq=10 ** 9, val_mesh_freq=10 ** 9,
        warm_up_end=4.0, anneal_end=0.0, learning_rate=r.learning_rate, learning_rate_alpha=r.learning_rate_alpha,
        renderer=types.SimpleNamespace(render=T.make_render(ref_params)), optimizer=torch.optim.Adam(ref_params, lr=r.learning_rate))
    for name in ("get_image_perm", "get_cos_anneal_ratio", "update_learning_rate"):
        setattr(ref, name, types.MethodType(ns[name], ref))
    torch.manual_seed(7)
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        ns["train"](ref)
    for i, q in enumerate(ref_params):
        arrays[f"{key}_param{i}_idx"], arrays[f"{key}_param{i}_val"] = param_sample(q, seed=i)
    return {"iter_step": ref.iter_step, "rec": wr_ref.rec, "final_lr": ref.optimizer.param_groups[0]["lr"], "n_params": len(ref_params),
            "param_shapes": [list(q.shape) for q in ref_params],
            "lr_printed": [l.split("lr=")[1] for l in buf.getvalue().splitlines() if "lr=" in l]}


def _train_clip_schedule(tmp):
    import test_train_loop_cpu as T
    from avatarclip_b200.runner import Runner
    from oracle.pin_sampling import reference_draws
    conf = open(os.path.join(ROOT, "tests", "runner_conf_sample.conf")).read().replace("./exp/CASE_NAME/demo", os.path.join(tmp, "clip"))
    for old, new in T.CLIP_CONF_EDITS:
        conf = conf.replace(old, new)
    p = os.path.join(tmp, "clip.conf")
    open(p, "w").write(conf)
    r = Runner(p, mode="train_clip", case="smpl", device="cpu")
    n = T.CLIP_STEPS
    body, face, back = torch.zeros(1, 4), torch.ones(1, 4), torch.full((1, 4), 2.0)
    draws = reference_draws(r.seed, n + 1, r.head_height, face=True, bg_aug=True, shading=True)
    prompt_lines = cut("main.py", 499, 507, "if self.use_face_prompt and iter_i % 4 == 0", "current_no_texture_text_encoding = self.encoded_text")
    sched = {"np": np}
    exec(cut("main.py", 571, 586, "def get_cos_anneal_ratio", "g['lr']"), sched)
    steps = []
    for i in range(n):
        s = types.SimpleNamespace(use_face_prompt=True, use_back_prompt=True, encoded_text=body, encoded_face_text=face, encoded_back_text=back)
        loc = dict(self=s, iter_i=i, is_front=draws[i]["is_front"])
        exec(prompt_lines, loc)
        sch = types.SimpleNamespace(iter_step=i, warm_up_end=5.0, end_iter=80, learning_rate_alpha=r.learning_rate_alpha,
                                    learning_rate=r.learning_rate, anneal_end=0.0,
                                    optimizer=types.SimpleNamespace(param_groups=[{"lr": None}]))
        sched["update_learning_rate"](sch)
        steps.append({"text": float(loc["current_text_encoding"][0, 0]),
                      "no_texture_text": float(loc["current_no_texture_text_encoding"][0, 0]),
                      "lr": sch.optimizer.param_groups[0]["lr"], "cos_anneal": float(sched["get_cos_anneal_ratio"](sch)),
                      "pose": np.asarray(draws[i]["pose"]).tolist(), "bg": int(draws[i]["choice_i"]),
                      "light": np.asarray(draws[i]["light_dir"]).astype(np.float32).tolist(), "ambience": draws[i]["ambience"]})
    return steps


# ------------------------------------------------------------------------------------------------ tests/test_validate_cpu.py
def _validate_image(tmp, extra_color, arrays):
    import cv2 as cv
    import test_validate_cpu as T
    ns = dict(np=np, torch=torch, os=os, cv=cv)
    exec(cut("main.py", 741, 820, "def validate_image(self, idx=-1, resolution_level=-1)", "normal_img[..., i])"), ns)
    base = os.path.join(tmp, f"vi{int(extra_color)}")
    ref_self = types.SimpleNamespace(dataset=T.FakeDataset(), iter_step=1234, batch_size=100, validate_resolution_level=1,
                                     use_white_bkgd=False, extra_color=extra_color, renderer=T.FakeRenderer(),
                                     base_exp_dir=base, get_cos_anneal_ratio=lambda: 1.0)
    ns["validate_image"](ref_self, idx=3, resolution_level=2)
    files = {}
    for d in sorted(os.listdir(base)):
        names = sorted(os.listdir(os.path.join(base, d)))
        files[d] = names
        for n in names:
            arrays[f"validate_image_{int(extra_color)}/{d}/{n}"] = cv.imread(os.path.join(base, d, n), cv.IMREAD_UNCHANGED)
    return files


def _validate_mesh(tmp, extra_color, arrays):
    import logging
    import test_validate_cpu as T
    captured = {}

    class Trimesh:                      # stand-in for the absent trimesh package: records what would be exported
        def __init__(self, vertices, triangles, vertex_colors=None):
            captured.update(vertices=np.asarray(vertices), triangles=np.asarray(triangles), colors=np.asarray(vertex_colors))

    tm = types.SimpleNamespace(Trimesh=Trimesh, exchange=types.SimpleNamespace(export=types.SimpleNamespace(
        export_mesh=lambda mesh, path, file_type=None: captured.update(path=path, file_type=file_type))))
    ns = dict(np=np, torch=torch, os=os, logging=logging, trimesh=tm, to8b=lambda x: (255 * np.clip(x, 0, 1)).astype(np.uint8))
    exec(cut("main.py", 850, 919, "def validate_mesh(self, world_space=False", "logging.info('End')"), ns)
    ds = T.FakeDataset()
    ds.object_bbox_min, ds.object_bbox_max = np.array([-1.01] * 3), np.array([1.01] * 3)
    ref_self = types.SimpleNamespace(dataset=ds, iter_step=77, batch_size=100, use_white_bkgd=False, extra_color=extra_color,
                                     renderer=T.MeshRenderer(), base_exp_dir=os.path.join(tmp, f"vm{int(extra_color)}"),
                                     get_cos_anneal_ratio=lambda: 1.0)
    saved_cuda = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self_, *a, **k: self_          # `.cuda()` (main.py:859,872): a device move
    try:
        ns["validate_mesh"](ref_self, resolution=64)
    finally:
        torch.Tensor.cuda = saved_cuda
    for k in ("vertices", "triangles", "colors"):
        arrays[f"validate_mesh_{int(extra_color)}_{k}"] = captured[k]
    return {"path": os.path.basename(captured["path"]), "file_type": captured["file_type"]}


def _cast_light(tmp, arrays):
    from torchvision import transforms
    import test_validate_cpu as T
    uns = dict(np=np, torch=torch)
    exec(cut("models/utils.py", 6, 27, "def norm_np_arr", "return _viewMatrix"), uns)
    exec(cut("models/utils.py", 59, 64, "def sphere_coord", "])"), uns)
    captured = {}
    ns = dict(np=np, torch=torch, os=os, transforms=transforms, lookat=uns["lookat"], sphere_coord=uns["sphere_coord"],
              imageio=types.SimpleNamespace(imwrite=lambda path, arr: captured.update(path=path, img=np.asarray(arr))),
              to8b=lambda x: (255 * np.clip(x, 0, 1)).astype(np.uint8))
    exec(cut("main.py", 634, 739, "def render_geometry_cast_light(self)", ")"), ns)
    ref_self = types.SimpleNamespace(dataset=T.CastLightDataset(), batch_size=500, head_height=0.55, renderer=T.FakeRenderer(),
                                     base_exp_dir=os.path.join(tmp, "cl"), get_cos_anneal_ratio=lambda: 1.0)
    os.makedirs(ref_self.base_exp_dir, exist_ok=True)
    saved_cuda = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self_, *a, **k: self_
    np.random.seed(21)
    try:
        ns["render_geometry_cast_light"](ref_self)
        next_ref = np.random.uniform()
    finally:
        torch.Tensor.cuda = saved_cuda
    arrays["cast_light_img"] = captured["img"]
    return {"path": os.path.basename(captured["path"]), "next_uniform": float(next_ref)}


def main():
    import tempfile
    if not os.path.isdir(REF):
        raise SystemExit(f"reference checkout not found at {REF}")
    if not make_ref.available():
        make_ref.stage(quiet=True)
    arrays, meta = {}, {}
    pin_confs()
    meta["fields"] = pin_fields()
    meta["dataset"] = pin_dataset()
    meta.update(pin_handoff(arrays))
    meta["checkpoint"] = pin_checkpoint()
    with tempfile.TemporaryDirectory() as tmp:
        meta["train_loop"] = {f"{mw}_{w}": _train_loop_case(os.path.join(tmp, f"tl_{mw}_{w}"), mw, w, arrays, f"train_loop_{mw}_{w}")
                              for mw, w in ((0.5, False), (0.0, True))}
        meta["train_clip"] = _train_clip_schedule(tmp)
        meta["validate_image"] = {str(int(e)): _validate_image(tmp, e, arrays) for e in (True, False)}
        meta["validate_mesh"] = {str(int(e)): _validate_mesh(tmp, e, arrays) for e in (True, False)}
        meta["cast_light"] = _cast_light(tmp, arrays)
    with open(os.path.join(GOLDEN, "host_mirrors.json"), "w") as f:
        json.dump(meta, f, indent=1)
    np.savez_compressed(os.path.join(GOLDEN, "host_mirrors.npz"), **arrays)
    print("[pin_host_mirrors] wrote", ", ".join(sorted(meta)))


if __name__ == "__main__":
    main()
