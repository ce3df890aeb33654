"""On-disk hand-off formats (avatarclip_b200/handoff.py), host side: the vertex-coloured binary PLY of Runner.validate_mesh
(main.py:913-916) and the camera matrices of the ShapeGen -> AppearanceGen directory (AvatarGen/ShapeGen/render.py:16-58)."""
import os

import numpy as np

from avatarclip_b200 import handoff

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_ply_round_trip_and_header(tmp_path):
    rng = np.random.RandomState(0)
    v = rng.randn(50, 3).astype(np.float32)
    f = rng.randint(0, 50, size=(80, 3)).astype(np.int64)
    c = rng.randint(0, 256, size=(50, 3)).astype(np.uint8)
    p = handoff.write_ply(str(tmp_path / "m.ply"), v, f, c)
    raw = open(p, "rb").read()
    head = raw[:raw.index(b"end_header\n")].decode("ascii").split("\n")
    assert head[:2] == ["ply", "format binary_little_endian 1.0"]
    assert "element vertex 50" in head and "element face 80" in head
    assert head.index("property uchar alpha") == head.index("property uchar red") + 3          # r g b a, like trimesh's export
    assert "property list uchar int vertex_indices" in head
    assert len(raw) == raw.index(b"end_header\n") + len(b"end_header\n") + 50 * (12 + 4) + 80 * (1 + 12)
    vv, ff, cc = handoff.read_ply(p)
    assert np.array_equal(vv, v) and np.array_equal(ff, f.astype(np.int32)) and np.array_equal(cc, c)
    p2 = handoff.write_ply(str(tmp_path / "plain.ply"), v, f)                                    # no colours
    vv, ff, cc = handoff.read_ply(p2)
    assert np.array_equal(vv, v) and np.array_equal(ff, f.astype(np.int32)) and cc is None
    p3 = handoff.write_ply(str(tmp_path / "empty.ply"), np.zeros((0, 3)), np.zeros((0, 3)), np.zeros((0, 3), dtype=np.uint8))
    vv, ff, cc = handoff.read_ply(p3)                                                            # an empty iso-surface
    assert vv.shape == (0, 3) and ff.shape == (0, 3) and cc.shape == (0, 3)


def test_hand_off_cameras():
    d = 2.2
    assert np.allclose(handoff.get_points_from_angles(d, 0, 0), [0, 0, -d])
    assert np.allclose(handoff.get_points_from_angles(d, 0, 90), [d, 0, 0], atol=1e-12)
    assert np.allclose(handoff.get_points_from_angles(d, 90, 0), [0, d, 0], atol=1e-12)
    eyes = [handoff.get_points_from_angles(d, e, a) for a in range(0, 360, 20) for e in range(-60, 60, 20)]
    assert len(eyes) == 108 and np.allclose([np.linalg.norm(e) for e in eyes], d)               # render.py:47-48
    for eye in eyes[::7]:
        m = handoff.lookat_inverse_view(eye, np.zeros(3), np.array([0.0, 1.0, 0.0]))
        R = m[:3, :3]
        assert np.allclose(R.T @ R, np.eye(3), atol=1e-12) and abs(np.linalg.det(R) - 1.0) < 1e-12
        assert np.allclose(m[:3, 3], eye) and np.allclose(m[3], [0, 0, 0, 1])
        assert np.allclose(R[:, 2], eye / np.linalg.norm(eye))                                    # camera looks down -z at the origin


def test_camera_matrix_equals_the_reference_lines():
    """handoff.lookat_inverse_view against what ShapeGen/render.py:16-30 (norm_np_arr + lookat), executed in place, returned for
    the same eyes (recorded by oracle/pin_host_mirrors.py)."""
    refs = iter(np.load(os.path.join(GOLDEN, "host_mirrors.npz"))["handoff_lookat"])
    for a in range(0, 360, 40):
        for e in (-60, -20, 0, 40):
            eye = handoff.get_points_from_angles(2.2, e, a)
            assert np.array_equal(next(refs), handoff.lookat_inverse_view(eye, np.array([0, 0, 0]), np.array([0, 1, 0])))


def test_read_obj_triangulates_and_strips_texture_indices(tmp_path):
    from avatarclip_b200.views import read_obj
    p = tmp_path / "t.obj"
    p.write_text("# comment\nv 0 0 0\nv 1 0 0\nv 1 1 0\nv 0 1 0\nvt 0 0\nvn 0 0 1\nf 1/1/1 2/1/1 3/1/1 4/1/1\nf 1 2 3\n")
    v, f = read_obj(str(p))
    assert v.shape == (4, 3) and v.dtype == np.float32
    assert f.tolist() == [[0, 1, 2], [0, 2, 3], [0, 1, 2]] and f.dtype == np.int32          # quad -> fan of two triangles


def test_read_obj_on_the_shipped_template():
    """dataset.template_obj of the shipped confs (main.py:292,316), the SMPL topology (6890 vertices / 13 776 triangles): the
    first 700 vertex lines of the shipped file and its face lines among them, verbatim (oracle/pin_host_mirrors.py)."""
    import json
    from avatarclip_b200.views import read_obj
    ref = json.load(open(os.path.join(GOLDEN, "host_mirrors.json")))["obj_sample"]
    path = os.path.join(GOLDEN, "zero_beta_smpl_sample.obj")
    v, f = read_obj(path)
    assert v.shape == (ref["n_verts"], 3) and f.shape == (ref["n_faces"], 3)
    assert f.min() == ref["face_min"] == 0 and f.max() == ref["face_max"]
    assert np.abs(v).max() < 1.5
    want_v = np.array([float(x) for l in open(path) if l.startswith("v ") for x in l.split()[1:]], dtype=np.float32).reshape(-1, 3)
    assert np.array_equal(v, want_v)
