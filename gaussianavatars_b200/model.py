"""Host-side stand-in for the splat model surface the path consumes (scene/gaussian_model.py:47-73,113-160 and
scene/flame_gaussian_model.py:117-154).  The licensed FLAME assets are absent (SURVEY.md 7.4-4), so
`MeshBoundGaussians` drives the same attributes from any (verts, faces) mesh:

    raw parameters : _xyz, _rotation, _scaling, _opacity, _features_dc, _features_rest, binding
    per-face frame : face_center, face_orien_mat, face_scaling, face_orien_quat  (update_mesh_properties)
    getters        : get_xyz / get_rotation / get_scaling / get_opacity / get_features   (eager torch -- the
                     reference route; the fused route never calls them)

It is what bench.py and the tests feed to `render()`; a real FlameGaussianModel exposes the same names, so the
renderer treats both alike.
"""
from __future__ import annotations

from typing import Callable, Dict, Optional

import torch
import torch.nn.functional as F


def face_frame(verts: torch.Tensor, faces: torch.Tensor, eps: float = 1e-20):
    """Per-face orthonormal frame, isotropic scale and centre (utils/graphics_utils.py:116-135,
    scene/flame_gaussian_model.py:139-143).  verts (V,3), faces (F,3) -> center (F,3), R (F,3,3) columns a0 a1 a2,
    scale (F,1)."""
    tri = verts[faces]
    v0, v1, v2 = tri[:, 0], tri[:, 1], tri[:, 2]

    def unit(v):
        return v / torch.sqrt(torch.clamp((v * v).sum(-1, keepdim=True), min=eps))

    e01, e02 = v1 - v0, v2 - v0
    a0 = unit(e01)
    a1 = unit(torch.cross(a0, e02, dim=-1))
    a2 = -unit(torch.cross(a1, a0, dim=-1))
    R = torch.stack((a0, a1, a2), dim=-1)
    s0 = torch.sqrt(torch.clamp((e01 * e01).sum(-1, keepdim=True), min=eps))
    s1 = (a2 * e02).sum(-1, keepdim=True).abs()
    return tri.mean(dim=1), R, (s0 + s1) / 2


def rotmat_to_quat_wxyz(R: torch.Tensor) -> torch.Tensor:
    """Unit quaternion (wxyz) of rotation matrices (N,3,3): largest-of-(diagonal, trace) branch, then normalise
    (the semantics of roma.rotmat_to_unitquat followed by quat_xyzw_to_wxyz; sign not canonicalised)."""
    m = R.reshape(-1, 3, 3)
    d0, d1, d2 = m[:, 0, 0], m[:, 1, 1], m[:, 2, 2]
    tr = d0 + d1 + d2
    choice = torch.stack((d0, d1, d2, tr), dim=1).argmax(dim=1)
    cand = []
    for i in range(3):
        j, k = (i + 1) % 3, (i + 2) % 3
        c = [None] * 4
        c[i] = 1 - tr + 2 * m[:, i, i]
        c[j] = m[:, j, i] + m[:, i, j]
        c[k] = m[:, k, i] + m[:, i, k]
        c[3] = m[:, k, j] - m[:, j, k]
        cand.append(torch.stack(c, dim=1))
    cand.append(torch.stack((m[:, 2, 1] - m[:, 1, 2], m[:, 0, 2] - m[:, 2, 0], m[:, 1, 0] - m[:, 0, 1], 1 + tr), 1))
    q = torch.zeros_like(cand[0])
    for c in range(4):
        q = torch.where((choice == c)[:, None], cand[c], q)
    q = q / q.norm(dim=1, keepdim=True)
    return torch.cat((q[:, 3:4], q[:, :3]), dim=1)


def quat_mul_wxyz(p: torch.Tensor, q: torch.Tensor) -> torch.Tensor:
    pw, pv = p[:, :1], p[:, 1:]
    qw, qv = q[:, :1], q[:, 1:]
    w = pw * qw - (pv * qv).sum(-1, keepdim=True)
    v = pw * qv + qw * pv + torch.cross(pv, qv, dim=-1)
    return torch.cat((w, v), dim=1)


class MeshBoundGaussians:
    def __init__(self, params: Dict[str, torch.Tensor], sh_degree: int, verts: Optional[torch.Tensor] = None,
                 faces: Optional[torch.Tensor] = None, pose_fn: Optional[Callable] = None, device="cuda",
                 requires_grad: bool = False, flame=None, flame_param: Optional[Dict[str, torch.Tensor]] = None):
        """flame / flame_param: a FusedFlameHead and its parameters (io.load_flame_param's layout): the mesh of
        `select_mesh_by_timestep(t)` is then `flame.mesh_at(flame_param, t)`; `verts` / `faces` default to the
        FLAME template and faces.  Otherwise the mesh is `pose_fn(verts, t)` (or `verts` itself)."""
        if (flame is None) != (flame_param is None):
            raise ValueError("flame and flame_param go together")
        if flame is not None:
            verts = flame.v_template if verts is None else verts
            faces = flame.faces if faces is None else faces
        self.flame, self.flame_param = flame, flame_param
        self.max_sh_degree = sh_degree
        self.active_sh_degree = sh_degree
        for k in ("_xyz", "_rotation", "_scaling", "_opacity", "_features_dc", "_features_rest"):
            t = params[k].to(device).contiguous()
            setattr(self, k, t.requires_grad_(requires_grad))
        b = params.get("binding")
        self.binding = None if b is None else b.to(device=device, dtype=torch.int32).contiguous()
        self.verts_rest = None if verts is None else verts.to(device)
        self.faces = None if faces is None else faces.to(device)
        self.pose_fn = pose_fn
        self.faces_i32 = None if faces is None else self.faces.to(torch.int32).contiguous()
        self.face_center = self.face_orien_mat = self.face_scaling = self._face_orien_quat = None
        self.verts = None
        self.timestep = None

    # ---- mesh ----
    def update_mesh_properties(self, verts: torch.Tensor):
        """scene/flame_gaussian_model.py:137-147.  On the GPU the frame is ONE library launch; the quaternion form is
        only materialised if the eager reference route asks for it (the fused route composes matrices)."""
        self.verts = verts
        # drop the previous frame (and the autograd graph hanging off it) BEFORE building the new one: a graph that is
        # still alive would hand its AccumulateGrad node for `verts` -- bound to the stream of an earlier step -- to the
        # new graph, which breaks CUDA-graph capture of the step (graph.py)
        self.face_center = self.face_orien_mat = self.face_scaling = None
        if verts.is_cuda:
            from .rasterizer import face_frame as face_frame_cuda

            self.face_center, self.face_orien_mat, self.face_scaling = face_frame_cuda(verts, self.faces_i32)
        else:
            self.face_center, self.face_orien_mat, self.face_scaling = face_frame(verts, self.faces)
        self._face_orien_quat = None

    @property
    def face_orien_quat(self):
        if self._face_orien_quat is None and self.face_orien_mat is not None:
            self._face_orien_quat = rotmat_to_quat_wxyz(self.face_orien_mat)
        return self._face_orien_quat

    def select_mesh_by_timestep(self, timestep: int):
        self.timestep = timestep
        if self.flame is not None:
            v = self.flame.mesh_at(self.flame_param, timestep)
        else:
            v = self.verts_rest if self.pose_fn is None else self.pose_fn(self.verts_rest, timestep)
        self.update_mesh_properties(v)

    # ---- getters: the reference route (eager) ----
    @property
    def get_scaling(self):
        s = torch.exp(self._scaling)
        return s if self.binding is None else s * self.face_scaling[self.binding.long()]

    @property
    def get_rotation(self):
        rot = F.normalize(self._rotation)
        if self.binding is None:
            return rot
        fq = F.normalize(self.face_orien_quat[self.binding.long()])
        return quat_mul_wxyz(fq, rot)

    @property
    def get_xyz(self):
        if self.binding is None:
            return self._xyz
        b = self.binding.long()
        # p_world = s_face R_face x_local + c_face per splat (SURVEY.md Appendix C "World transform")
        rotated = torch.einsum("pij,pj->pi", self.face_orien_mat[b], self._xyz)
        return torch.addcmul(self.face_center[b], rotated, self.face_scaling[b])

    @property
    def get_features(self):
        return torch.cat((self._features_dc, self._features_rest), dim=1)

    @property
    def get_opacity(self):
        return torch.sigmoid(self._opacity)

    def parameters(self):
        return [self._xyz, self._rotation, self._scaling, self._opacity, self._features_dc, self._features_rest]
