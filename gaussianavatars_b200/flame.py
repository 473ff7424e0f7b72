"""FLAME head on the GPU: blendshapes + linear blend skinning and their backward as library launches
(include/gab200_rasterizer.h gab200_flame_*).

    head = FusedFlameHead.from_flame_head(gaussians.flame_model)    # adopt a built reference FlameHead
    gaussians.flame_model = head                                    # drop-in: same forward signature and outputs
    verts = head.mesh_at(flame_param, timestep)                     # (V,3), differentiable into the (T,k) tables

The model arrays are inputs (the licensed FLAME assets are not part of this project): a FlameHead the user already
built, or the same arrays in FlameHead's layout.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict

import torch
import torch.nn as nn

from . import _native as N

NUM_JOINTS = 5
# flame_param keys of the per-timestep tables, in the order of the kernel's arguments (FlameGaussianModel)
TABLE_KEYS = ("expr", "rotation", "neck_pose", "jaw_pose", "eyes_pose", "translation")


def _cuda_f32(t: torch.Tensor, name: str, device) -> torch.Tensor:
    if t.device.type != "cuda":
        raise RuntimeError("gaussianavatars_b200 has no CPU path: tensors must be CUDA tensors")
    if t.device != device:
        raise ValueError(f"{name} is on {t.device}, the FLAME model on {device}")
    return t if (t.dtype == torch.float32 and t.is_contiguous()) else t.float().contiguous()


class _FlameFn(torch.autograd.Function):
    """verts, verts_cano of one call; gradients are added into row `row` of zeroed (T,k) tables."""

    @staticmethod
    def forward(ctx, head, row, shape, expr, rotation, neck, jaw, eyes, translation, static_offset):
        device = head.v_template.device
        V, T = head.num_verts, expr.shape[0]
        a = head._model_args(T)
        a.row = None if row is None else row.data_ptr()
        a.shape = N.ptr(shape)
        a.expr, a.rotation, a.neck, a.jaw, a.eyes, a.translation = (t.data_ptr() for t in
                                                                     (expr, rotation, neck, jaw, eyes, translation))
        a.static_offset = N.ptr(static_offset)
        verts = torch.empty((V, 3), dtype=torch.float32, device=device)
        cano = torch.empty((V, 3), dtype=torch.float32, device=device)
        ws = torch.empty(head._workspace_bytes, dtype=torch.uint8, device=device)
        a.verts, a.verts_cano, a.workspace = verts.data_ptr(), cano.data_ptr(), ws.data_ptr()
        with torch.cuda.device(device):
            stream = torch.cuda.current_stream(device).cuda_stream
            N.check(N.lib().gab200_flame_forward(C.byref(a), C.c_void_p(stream)), "gab200_flame_forward")
        ctx.args, ctx.ws = a, ws
        ctx.keep = (row, shape, expr, rotation, neck, jaw, eyes, translation, static_offset)
        ctx.mark_non_differentiable(cano)
        return verts, cano

    @staticmethod
    def backward(ctx, g_verts, g_cano):
        inputs = ctx.keep[1:]
        want = ctx.needs_input_grad[2:]
        grads = [None] * len(inputs)
        if g_verts is None or not any(want):
            return (None, None, *grads)
        sizes = [t.numel() if (w and t is not None) else 0 for t, w in zip(inputs, want)]
        flat = torch.zeros(sum(sizes), dtype=torch.float32, device=g_verts.device)   # one memset for all tables
        off = 0
        for i, (t, n) in enumerate(zip(inputs, sizes)):
            if n:
                grads[i] = flat[off:off + n].view(t.shape)
                off += n
        a = ctx.args
        (a.grad_shape, a.grad_expr, a.grad_rotation, a.grad_neck, a.grad_jaw, a.grad_eyes, a.grad_translation,
         a.grad_static_offset) = (N.ptr(g) for g in grads)
        g = g_verts if (g_verts.dtype == torch.float32 and g_verts.is_contiguous()) else g_verts.float().contiguous()
        with torch.cuda.device(g.device):
            stream = torch.cuda.current_stream(g.device).cuda_stream
            N.check(N.lib().gab200_flame_backward(C.byref(a), g.data_ptr(), C.c_void_p(stream)), "gab200_flame_backward")
        return (None, None, *grads)


class FusedFlameHead(nn.Module):
    """FLAME with the buffers of the reference FlameHead (v_template, shapedirs, posedirs, J_regressor, parents,
    lbs_weights, faces) plus the joint arrays precomputed from them (J_template, J_shapedirs).  `forward` has
    FlameHead.forward's signature; the mesh is computed by the library's FLAME kernels."""

    def __init__(self, v_template, shapedirs, posedirs, J_regressor, parents, lbs_weights, faces, n_shape: int,
                 n_expr: int):
        super().__init__()
        v_template = torch.as_tensor(v_template)
        V = v_template.shape[0]
        NB = int(n_shape) + int(n_expr)
        J = torch.as_tensor(J_regressor).shape[0]
        if J != NUM_JOINTS:
            raise ValueError(f"FLAME has {NUM_JOINTS} joints (global, neck, jaw, eyes); J_regressor has {J} rows")
        expect = {"v_template": (v_template, (V, 3)), "shapedirs": (shapedirs, (V, 3, NB)),
                  "posedirs": (posedirs, ((J - 1) * 9, 3 * V)), "J_regressor": (J_regressor, (J, V)),
                  "lbs_weights": (lbs_weights, (V, J)), "parents": (parents, (J,))}
        for name, (t, shp) in expect.items():
            if tuple(torch.as_tensor(t).shape) != shp:
                raise ValueError(f"{name} has shape {tuple(torch.as_tensor(t).shape)}, expected {shp}")
        par = torch.as_tensor(parents).long()
        if par[0] != -1 or any(not (0 <= int(par[j]) < j) for j in range(1, J)):
            raise ValueError(f"parents must be -1 followed by indices of earlier joints, got {par.tolist()}")
        faces = torch.as_tensor(faces)
        if faces.ndim != 2 or faces.shape[1] != 3:
            raise ValueError("faces must be (F,3)")
        f32 = lambda t: torch.as_tensor(t).detach().to(torch.float32).contiguous()  # noqa: E731
        self.n_shape_params, self.n_expr_params = int(n_shape), int(n_expr)
        self.dtype = torch.float32
        self.register_buffer("v_template", f32(v_template))
        self.register_buffer("shapedirs", f32(shapedirs))
        self.register_buffer("posedirs", f32(posedirs))
        self.register_buffer("J_regressor", f32(J_regressor))
        self.register_buffer("parents", par.clone())
        self.register_buffer("lbs_weights", f32(lbs_weights))
        self.register_buffer("faces", faces.long().clone(), persistent=False)
        jr = torch.as_tensor(J_regressor).detach().double()
        self.register_buffer("J_template", (jr @ torch.as_tensor(v_template).detach().double()).float())
        self.register_buffer("J_shapedirs", torch.einsum("jv,vkl->jkl", jr, torch.as_tensor(shapedirs).detach().double())
                             .float().contiguous())
        self.register_buffer("parents_i32", par.to(torch.int32), persistent=False)
        self._rows = {}
        self._workspace_bytes = 0

    @classmethod
    def from_flame_head(cls, head) -> "FusedFlameHead":
        """Adopts the buffers of a built reference FlameHead (teeth included when it added them) on the head's device.
        Attributes this module does not own (mask, verts_uvs, textures_idx, ...) are read from `head`."""
        new = cls(head.v_template, head.shapedirs, head.posedirs, head.J_regressor, head.parents, head.lbs_weights,
                  head.faces, head.n_shape_params, head.n_expr_params)
        object.__setattr__(new, "_origin", head)   # not a submodule: its buffers are not ours to save or move
        return new.to(head.v_template.device)

    def __getattr__(self, name):
        try:
            return super().__getattr__(name)
        except AttributeError:
            origin = self.__dict__.get("_origin")
            if origin is None:
                raise
            return getattr(origin, name)

    @property
    def num_verts(self) -> int:
        return self.v_template.shape[0]

    def _model_args(self, T: int) -> N.FlameArgs:
        if self.v_template.device.type != "cuda":
            raise RuntimeError("gaussianavatars_b200 has no CPU path: move the FLAME model to a CUDA device")
        V = self.num_verts
        if not self._workspace_bytes:
            self._workspace_bytes = int(N.lib().gab200_flame_workspace_bytes(V, self.n_shape_params, self.n_expr_params))
        a = N.FlameArgs()
        a.abi_version, a.V, a.n_shape, a.n_expr, a.J, a.T = N.ABI_VERSION, V, self.n_shape_params, self.n_expr_params, \
            NUM_JOINTS, int(T)
        for name in ("v_template", "shapedirs", "posedirs", "J_regressor", "lbs_weights", "J_template", "J_shapedirs"):
            setattr(a, name, getattr(self, name).data_ptr())
        a.parents = self.parents_i32.data_ptr()
        return a

    def _apply_fn(self, row, shape, tables, static_offset):
        device = self.v_template.device
        if device.type != "cuda":
            raise RuntimeError("gaussianavatars_b200 has no CPU path: move the FLAME model to a CUDA device")
        T = tables[0].shape[0]
        widths = (self.n_expr_params, 3, 3, 3, 6, 3)
        for t, w, name in zip(tables, widths, ("expr", "rotation", "neck", "jaw", "eyes", "translation")):
            if t.ndim != 2 or t.shape[1] != w or t.shape[0] != T:
                raise ValueError(f"{name} has shape {tuple(t.shape)}, expected ({T}, {w})")
        tables = [_cuda_f32(t, name, device) for t, name in zip(tables, ("expr", "rotation", "neck", "jaw", "eyes",
                                                                           "translation"))]
        if shape is not None:
            if shape.numel() != self.n_shape_params:
                raise ValueError(f"shape has {shape.numel()} values, the model {self.n_shape_params}")
            shape = _cuda_f32(shape.reshape(-1), "shape", device)
        if static_offset is not None:
            if static_offset.numel() != 3 * self.num_verts:
                raise ValueError(f"static_offset has shape {tuple(static_offset.shape)}, expected (1, {self.num_verts}, 3)")
            static_offset = _cuda_f32(static_offset.reshape(self.num_verts, 3), "static_offset", device)
        return _FlameFn.apply(self, row, shape, *tables, static_offset)

    def forward(
        self,
        shape,
        expr,
        rotation,
        neck,
        jaw,
        eyes,
        translation,
        zero_centered_at_root_node=False,  # otherwise, zero centered at the face
        return_landmarks=True,
        return_verts_cano=False,
        static_offset=None,
        dynamic_offset=None,
    ):
        """FlameHead.forward for a batch of one: verts (1,V,3) [, verts_cano (1,V,3)].  `dynamic_offset` is accepted
        and ignored, as in FlameHead; verts_cano is not differentiable."""
        if return_landmarks:
            raise NotImplementedError("FusedFlameHead computes no landmarks: call it with return_landmarks=False")
        if zero_centered_at_root_node:
            raise NotImplementedError("FusedFlameHead supports zero_centered_at_root_node=False only")
        if shape.shape[0] != 1 or expr.shape[0] != 1:
            raise NotImplementedError("FusedFlameHead poses one mesh per call (batch size 1)")
        verts, cano = self._apply_fn(None, shape, (expr, rotation, neck, jaw, eyes, translation), static_offset)
        if return_verts_cano:
            return [verts[None], cano[None]]
        return verts[None]

    def row_index(self, timestep) -> torch.Tensor:
        """A device int32 tensor holding `timestep` (cached per value)."""
        if isinstance(timestep, torch.Tensor):
            if timestep.device.type != "cuda" or timestep.dtype != torch.int32 or timestep.numel() != 1:
                raise ValueError("a tensor timestep must be a one-element int32 CUDA tensor")
            return timestep
        t = int(timestep)
        key = (self.v_template.device, t)
        r = self._rows.get(key)
        if r is None:
            r = torch.tensor([t], dtype=torch.int32, device=self.v_template.device)
            self._rows[key] = r
        return r

    def mesh_at(self, flame_param: Dict[str, torch.Tensor], timestep) -> torch.Tensor:
        """Posed vertices (V,3) of `flame_param` (the layout of io.load_flame_param) at `timestep` (an int, or a
        one-element int32 CUDA tensor read by the kernel -- what a CUDA graph replays).  Differentiable into every
        (T,k) table and into shape / static_offset: their gradients are dense with one non-zero row, like those of
        FlameGaussianModel's `flame_param[k][[t]]`."""
        tables = [flame_param[k] for k in TABLE_KEYS]
        if not isinstance(timestep, torch.Tensor) and not (0 <= int(timestep) < tables[0].shape[0]):
            raise IndexError(f"timestep {timestep} is out of range for {tables[0].shape[0]} frames")
        verts, _ = self._apply_fn(self.row_index(timestep), flame_param.get("shape"), tables,
                                  flame_param.get("static_offset"))
        return verts
