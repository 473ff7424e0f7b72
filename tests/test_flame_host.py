"""CPU: the FLAME surface without launching anything -- the ctypes mirror of gab200_flame_args matches the C layout,
FusedFlameHead.forward keeps FlameHead.forward's signature, and malformed models / calls are rejected."""
import ctypes as C
import inspect
import json
import os
import subprocess

import pytest
import torch

from gaussianavatars_b200 import FusedFlameHead
from gaussianavatars_b200.synthetic import flame_like_model

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
HEADER = os.path.join(ROOT, "include", "gab200_rasterizer.h")


@pytest.fixture(scope="module")
def small():
    return flame_like_model(1, n_shape=6, n_expr=4, n_lat=6, n_lon=8)


def _head(m, **over):
    a = dict(m, **over)
    return FusedFlameHead(a["v_template"], a["shapedirs"], a["posedirs"], a["J_regressor"], a["parents"],
                          a["lbs_weights"], a["faces"], a["n_shape"], a["n_expr"])


def test_flame_args_ctypes_mirror_matches_the_c_layout(tmp_path):
    from gaussianavatars_b200 import _native as N

    ct = N.FlameArgs
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', "int main(){",
             'printf("size %zu\\n", sizeof(gab200_flame_args));']
    for fname, _ in ct._fields_:
        lines.append(f'printf("{fname} %zu\\n", offsetof(gab200_flame_args, {fname}));')
    lines.append("return 0;}")
    src = tmp_path / "probe.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "probe"
    subprocess.run(["/usr/bin/gcc", str(src), "-o", str(exe)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    assert int(got["size"]) == C.sizeof(ct)
    for fname, _ in ct._fields_:
        assert int(got[fname]) == getattr(ct, fname).offset, fname


def test_workspace_size_is_positive_and_grows_with_the_model():
    from gaussianavatars_b200 import _native as N

    small, big = N.lib().gab200_flame_workspace_bytes(100, 6, 4), N.lib().gab200_flame_workspace_bytes(5143, 300, 100)
    assert 0 < small < big and big % 256 == 0


def test_forward_signature_is_the_reference_one():
    with open(os.path.join(ROOT, "tests", "golden", "flame_facts.json")) as f:
        facts = json.load(f)
    assert str(inspect.signature(FusedFlameHead.forward)) == facts["FlameHead.forward"]


def test_model_buffers_and_precomputed_joints(small):
    h = _head(small)
    names = dict(h.named_buffers())
    for k in ("v_template", "shapedirs", "posedirs", "J_regressor", "parents", "lbs_weights", "faces", "J_template",
              "J_shapedirs"):
        assert k in names, k
    jr = small["J_regressor"].double()
    assert torch.allclose(h.J_template.double(), jr @ small["v_template"].double(), atol=1e-7)
    assert torch.allclose(h.J_shapedirs.double(), torch.einsum("jv,vkl->jkl", jr, small["shapedirs"].double()), atol=1e-9)


def test_malformed_models_are_rejected(small):
    V = small["v_template"].shape[0]
    with pytest.raises(ValueError, match="5 joints"):
        _head(small, J_regressor=torch.zeros(4, V))
    with pytest.raises(ValueError, match="shapedirs"):
        _head(small, shapedirs=small["shapedirs"][:, :, :-1])
    with pytest.raises(ValueError, match="posedirs"):
        _head(small, posedirs=small["posedirs"][:27])
    with pytest.raises(ValueError, match="lbs_weights"):
        _head(small, lbs_weights=small["lbs_weights"][:-1])
    with pytest.raises(ValueError, match="parents"):
        _head(small, parents=torch.tensor([-1, 0, 3, 1, 1]))


def test_calls_outside_the_supported_surface_are_rejected(small):
    h = _head(small)
    z = lambda *s: torch.zeros(*s)  # noqa: E731
    call = (z(1, 6), z(1, 4), z(1, 3), z(1, 3), z(1, 3), z(1, 6), z(1, 3))
    with pytest.raises(NotImplementedError, match="landmarks"):
        h(*call)   # FlameHead's default return_landmarks=True
    with pytest.raises(NotImplementedError, match="zero_centered_at_root_node"):
        h(*call, zero_centered_at_root_node=True, return_landmarks=False)
    with pytest.raises(NotImplementedError, match="batch size 1"):
        h(z(2, 6), z(2, 4), z(2, 3), z(2, 3), z(2, 3), z(2, 6), z(2, 3), return_landmarks=False)
    with pytest.raises(RuntimeError, match="no CPU path"):
        h(*call, return_landmarks=False, return_verts_cano=True)
    fp = {"shape": z(6), "expr": z(5, 4), "rotation": z(5, 3), "neck_pose": z(5, 3), "jaw_pose": z(5, 3),
          "eyes_pose": z(5, 6), "translation": z(5, 3)}
    with pytest.raises(IndexError):
        h.mesh_at(fp, 5)
    with pytest.raises(RuntimeError, match="no CPU path"):
        h.mesh_at(fp, 1)


def test_from_flame_head_delegates_attributes_it_does_not_own(small):
    src = _head(small)
    src.mask = "region masks"          # stands in for FlameHead.mask / verts_uvs
    h = FusedFlameHead.from_flame_head(src)
    assert h.mask == "region masks" and h.n_shape_params == 6 and h.num_verts == small["v_template"].shape[0]
    assert not any(n.startswith("_origin") for n, _ in h.named_buffers())
    with pytest.raises(AttributeError):
        h.no_such_attribute
