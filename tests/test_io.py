"""CPU: the splat PLY format (gaussianavatars_b200/io.py) against the reference's writer/reader
(scene/gaussian_model.py:234-332) and against samples of the demo avatar it ships (tests/golden/make_golden_demo.py)."""
import hashlib
import json
import os

import numpy as np
import pytest
import torch

from gaussianavatars_b200 import io as gio

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
FACTS = json.load(open(os.path.join(GOLDEN, "reference_facts.json")))
DEMO = os.path.join(GOLDEN, "demo_point_cloud_sample.ply")   # media/306/point_cloud.ply: a sample of its records
# sha256 of the 1555-byte header of media/306/point_cloud.ply (89,021 vertices, 63 float properties incl. binding_0),
# recorded from the real file: pins `ply_header` to plyfile's output without shipping the asset
DEMO_HEADER_SHA256 = "4f7c89da20e1671bf40dae12e75a21aeabe7c91ec9cf9ec980479f234363cbda"


def _params(P, deg, seed=0, binding=True):
    g = torch.Generator().manual_seed(seed)
    n_rest = (deg + 1) ** 2 - 1
    d = {"_xyz": torch.randn(P, 3, generator=g), "_features_dc": torch.randn(P, 1, 3, generator=g),
         "_features_rest": torch.randn(P, n_rest, 3, generator=g), "_opacity": torch.randn(P, 1, generator=g),
         "_scaling": torch.randn(P, 3, generator=g), "_rotation": torch.randn(P, 4, generator=g),
         "binding": torch.randint(0, 10144, (P,), generator=g, dtype=torch.int32) if binding else None}
    return d


@pytest.mark.parametrize("P,deg,binding", [(257, 3, True), (64, 3, False), (5, 0, True), (0, 3, True), (33, 1, False)])
def test_save_then_load_is_the_identity(tmp_path, P, deg, binding):
    d = _params(P, deg, binding=binding)
    path = str(tmp_path / "sub" / "point_cloud.ply")
    gio.save_ply(path, d)
    back = gio.load_ply(path, max_sh_degree=deg)
    for k, v in d.items():
        if v is None:
            assert back[k] is None
        else:
            assert back[k].dtype == v.dtype and back[k].shape == v.shape, k
            assert torch.equal(back[k], v), k
            assert back[k].is_contiguous()
    size = os.path.getsize(path)
    names = gio.attribute_names(3 * ((deg + 1) ** 2 - 1), binding)
    assert size == len(gio.ply_header(P, names)) + 4 * len(names) * P


def test_record_layout_is_the_reference_writers():
    """x y z, three zero normals, SH channel-major, opacity, scale, rot, binding as float (scene/gaussian_model.py:253-275)."""
    d = _params(3, 3, seed=1)
    raw = None
    import tempfile
    with tempfile.TemporaryDirectory() as t:
        gio.save_ply(os.path.join(t, "a.ply"), d)
        raw = open(os.path.join(t, "a.ply"), "rb").read()
    names = gio.attribute_names(45, True)
    assert names[:9] == ["x", "y", "z", "nx", "ny", "nz", "f_dc_0", "f_dc_1", "f_dc_2"]
    assert names[9] == "f_rest_0" and names[53] == "f_rest_44" and names[54:] == [
        "opacity", "scale_0", "scale_1", "scale_2", "rot_0", "rot_1", "rot_2", "rot_3", "binding_0"]
    hdr = gio.ply_header(3, names)
    assert raw.startswith(hdr) and hdr.endswith(b"end_header\n")
    table = np.frombuffer(raw[len(hdr):], dtype="<f4").reshape(3, 63)
    assert np.array_equal(table[:, 0:3], d["_xyz"].numpy()) and not table[:, 3:6].any()
    # f_rest_{c*15+k} = coefficient k+1 of channel c
    assert table[1, 9 + 2 * 15 + 4] == d["_features_rest"][1, 4, 2].item()
    assert table[2, 6 + 1] == d["_features_dc"][2, 0, 1].item()
    assert np.array_equal(table[:, 62], d["binding"].numpy().astype(np.float32))


def test_header_matches_the_reference_demo_file_byte_for_byte():
    hdr = gio.ply_header(89021, gio.attribute_names(45, True))
    assert len(hdr) == 1555                                   # SURVEY.md 8(d) config 2: "header 1555 B, 63 f32 props"
    assert hashlib.sha256(hdr).hexdigest() == DEMO_HEADER_SHA256


def test_reader_accepts_reordered_and_foreign_properties_and_rejects_other_formats(tmp_path):
    # a file whose properties come in another order, with a double and a uchar column mixed in and a second element
    P = 7
    dt = np.dtype([("opacity", "<f4"), ("z", "<f8"), ("flag", "u1"), ("y", "<f4"), ("x", "<f4")] +
                  [(n, "<f4") for n in ["rot_3", "rot_1", "rot_0", "rot_2", "scale_2", "scale_0", "scale_1",
                                        "f_dc_2", "f_dc_0", "f_dc_1"]])
    rec = np.zeros(P, dtype=dt)
    rng = np.random.default_rng(0)
    for n in dt.names:
        rec[n] = rng.integers(0, 200, P) if n == "flag" else rng.standard_normal(P)
    hdr = "ply\nformat binary_little_endian 1.0\ncomment made by hand\nelement vertex 7\n"
    kinds = {"<f4": "float", "<f8": "double", "u1": "uchar", "|u1": "uchar"}
    hdr += "".join(f"property {kinds[dt[n].str]} {n}\n" for n in dt.names)
    hdr += "element face 0\nproperty list uchar int vertex_indices\nend_header\n"
    path = tmp_path / "odd.ply"
    path.write_bytes(hdr.encode() + rec.tobytes())
    d = gio.load_ply(str(path), max_sh_degree=0)
    assert torch.equal(d["_xyz"], torch.tensor(np.stack([rec["x"], rec["y"], rec["z"].astype(np.float32)], 1).copy()))
    assert torch.equal(d["_rotation"][:, 2], torch.tensor(np.ascontiguousarray(rec["rot_2"]))) and d["binding"] is None
    assert d["_features_rest"].shape == (P, 0, 3)
    with pytest.raises(ValueError, match="f_rest"):
        gio.load_ply(str(path), max_sh_degree=3)
    asc = tmp_path / "ascii.ply"
    asc.write_bytes(b"ply\nformat ascii 1.0\nelement vertex 0\nproperty float x\nend_header\n")
    with pytest.raises(ValueError, match="binary_little_endian"):
        gio.load_ply(str(asc))
    bad = tmp_path / "bad.ply"
    bad.write_bytes(b"plx\n")
    with pytest.raises(ValueError):
        gio.load_ply(str(bad))


def test_loaded_parameters_drive_the_bound_model():
    """The dict is what MeshBoundGaussians takes (the reference: FlameGaussianModel.load_ply + binding)."""
    from gaussianavatars_b200 import synthetic as syn
    from gaussianavatars_b200.model import MeshBoundGaussians
    import tempfile

    verts, faces = syn.head_mesh()
    params = syn.avatar_splats(500, n_faces=faces.shape[0], seed=3, sh_degree=3)
    with tempfile.TemporaryDirectory() as t:
        gio.save_ply(os.path.join(t, "pc.ply"), params)
        back = gio.load_ply(os.path.join(t, "pc.ply"))
    a = MeshBoundGaussians(params, 3, verts, faces, device=torch.device("cpu"))
    b = MeshBoundGaussians(back, 3, verts, faces, device=torch.device("cpu"))
    a.update_mesh_properties(a.verts_rest)
    b.update_mesh_properties(b.verts_rest)
    assert torch.equal(a.get_xyz, b.get_xyz) and torch.equal(a.get_features, b.get_features)
    assert torch.equal(a.binding, b.binding)


def test_demo_avatar_of_the_reference_round_trips_byte_for_byte(tmp_path):
    facts = FACTS["point_cloud"]
    raw = open(DEMO, "rb").read()
    hdr = raw[:raw.index(b"end_header\n") + len(b"end_header\n")]
    # the sample sits under the demo file's own header, vertex count aside
    full = hdr.replace(b"element vertex %d\n" % facts["vertices"], b"element vertex %d\n" % facts["source_vertices"])
    assert facts["source_vertices"] == 89021 and hashlib.sha256(full).hexdigest() == DEMO_HEADER_SHA256
    d = gio.load_ply(DEMO)
    P = d["_xyz"].shape[0]
    assert P == facts["vertices"] and d["_features_rest"].shape == (P, 15, 3) and d["binding"].dtype == torch.int32
    assert (facts["source_binding_min"], facts["source_binding_max"]) == (0, 10143)   # SURVEY.md 8(d) config 2
    assert int(d["binding"].min()) == facts["binding_min"] and int(d["binding"].max()) == facts["binding_max"]
    assert abs(float(torch.sigmoid(d["_opacity"].double()).mean()) - facts["opacity_sigmoid_mean"]) < 1e-9
    out = tmp_path / "again.ply"
    gio.save_ply(str(out), d)
    h1, h2 = hashlib.sha256(), hashlib.sha256()
    h1.update(open(DEMO, "rb").read())
    h2.update(out.read_bytes())
    assert h1.hexdigest() == h2.hexdigest()


# ------------------------------------------------------------------------------------------------------------
# flame_param.npz
# ------------------------------------------------------------------------------------------------------------
DEMO_NPZ = os.path.join(GOLDEN, "demo_flame_param_sample.npz")   # media/306/flame_param.npz: frames and vertices cut


def _fake_flame(T, V=37, seed=0):
    g = torch.Generator().manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=g)  # noqa: E731
    return {"shape": r(300), "expr": r(T, 100), "rotation": r(T, 3), "neck_pose": r(T, 3), "jaw_pose": r(T, 3),
            "eyes_pose": r(T, 6), "translation": r(T, 3), "static_offset": r(1, V, 3), "dynamic_offset": r(T, V, 3)}


@pytest.mark.parametrize("mmap", [True, False])
def test_flame_param_round_trip_and_motion_override(tmp_path, mmap):
    fp = _fake_flame(5)
    p = gio.save_flame_param(str(tmp_path / "a" / "point_cloud.ply"), fp)
    assert p.endswith("flame_param.npz") and os.path.exists(p)
    back = gio.load_flame_param(p, mmap=mmap)
    assert list(back) == list(fp)
    for k in fp:
        assert back[k].dtype == torch.float32 and torch.equal(back[k], fp[k]), k
    # np.load agrees (the writer is np.savez, the reference's)
    z = np.load(p)
    assert z.files == list(fp) and all(np.array_equal(z[k], fp[k].numpy()) for k in fp)
    # motion sequence: static entries kept, dynamic ones replaced, non-float32 entries of the motion file ignored
    mo = _fake_flame(9, seed=1)
    mp = str(tmp_path / "motion.npz")
    np.savez(mp, **{k: v.numpy() for k, v in mo.items()}, frame_id=np.arange(9))
    mixed = gio.load_flame_param(p, motion_path=mp, mmap=mmap)
    assert set(mixed) == set(fp)
    for k in gio.FLAME_STATIC_KEYS:
        assert torch.equal(mixed[k], fp[k])
    for k in gio.FLAME_DYNAMIC_KEYS:
        assert torch.equal(mixed[k], mo[k]) and mixed[k].shape[0] == 9


def test_flame_param_of_the_demo_avatar(tmp_path):
    """media/306/flame_param.npz: mapped in place == np.load, and re-saved member by member byte-identical (the .npy
    payloads; zip timestamps differ between any two np.savez calls)."""
    import zipfile

    facts = FACTS["flame_param"]
    T, V = facts["frames"], facts["vertices"]
    fp = gio.load_flame_param(DEMO_NPZ)
    assert {k: list(v.shape) for k, v in fp.items()} == facts["shapes"]
    assert fp["expr"].shape == (T, 100) and fp["static_offset"].shape == (1, V, 3) and fp["shape"].shape == (300,)
    assert fp["dynamic_offset"].shape == (T, V, 3) and fp["eyes_pose"].shape == (T, 6)
    z = np.load(DEMO_NPZ)
    small = [k for k in z.files if k != "dynamic_offset"]
    for k in small:
        assert np.array_equal(fp[k].numpy(), z[k]), k
    out = gio.save_flame_param(str(tmp_path / "flame_param.npz"), {k: fp[k] for k in small})
    with zipfile.ZipFile(DEMO_NPZ) as a, zipfile.ZipFile(out) as b:
        assert [i.filename for i in b.infolist()] == [k + ".npy" for k in small]
        for k in small:
            assert a.read(k + ".npy") == b.read(k + ".npy"), k
