"""FLAME forward restated in plain torch (test infrastructure): blendshapes, Rodrigues with the reference's epsilon
placement, pose blendshapes, kinematic chain and linear blend skinning, written from the equations of
gaussianavatars_b200/csrc/flame.cu's header.  Differentiable under autograd in every float input; run it in float64
for a reference, in float32 for an eager arm of the same maths."""
from __future__ import annotations

import torch


def rodrigues(r: torch.Tensor) -> torch.Tensor:
    """(N,3) axis-angle -> (N,3,3): angle = |r + 1e-8| (per component), direction = r / angle."""
    a = torch.linalg.vector_norm(r + 1e-8, dim=1, keepdim=True)
    d = r / a
    x, y, z = d[:, 0], d[:, 1], d[:, 2]
    o = torch.zeros_like(x)
    K = torch.stack((o, -z, y, z, o, -x, -y, x, o), dim=1).view(-1, 3, 3)
    eye = torch.eye(3, dtype=r.dtype, device=r.device)
    return eye + torch.sin(a)[:, :, None] * K + (1 - torch.cos(a))[:, :, None] * (K @ K)


def flame_forward(model, shape, expr, rotation, neck, jaw, eyes, translation, static_offset=None):
    """model: dict of v_template (V,3), shapedirs (V,3,NB), posedirs (36,3V), J_regressor (5,V), parents (5,),
    lbs_weights (V,5).  Parameters of one mesh: shape (n_shape,), expr (n_expr,), rotation / neck / jaw /
    translation (3,), eyes (6,), static_offset (V,3) or None.  Returns verts (V,3), verts_cano (V,3)."""
    dt = expr.dtype
    vt = model["v_template"].to(dt)
    V = vt.shape[0]
    betas = torch.cat((shape.reshape(-1), expr.reshape(-1)))
    v_shaped = vt + torch.einsum("vkl,l->vk", model["shapedirs"].to(dt), betas)
    if static_offset is not None:
        v_shaped = v_shaped + static_offset.reshape(V, 3)
    Jr = model["J_regressor"].to(dt)
    J = Jr @ v_shaped                                                     # (5,3)
    pose = torch.cat((rotation.reshape(-1), neck.reshape(-1), jaw.reshape(-1), eyes.reshape(-1))).view(-1, 3)
    R = rodrigues(pose)                                                   # (5,3,3)
    eye = torch.eye(3, dtype=dt, device=vt.device)
    pose_feature = (R[1:] - eye).reshape(-1)                              # (36,)
    v_posed = v_shaped + (pose_feature @ model["posedirs"].to(dt)).view(V, 3)
    parents = [int(p) for p in model["parents"]]
    Rg, tg = [R[0]], [J[0]]
    for j in range(1, len(parents)):
        p = parents[j]
        Rg.append(Rg[p] @ R[j])
        tg.append(Rg[p] @ (J[j] - J[p]) + tg[p])
    Rg, tg = torch.stack(Rg), torch.stack(tg)
    A = torch.cat((Rg, (tg - torch.einsum("jrc,jc->jr", Rg, J))[:, :, None]), dim=2)   # (5,3,4)
    T = torch.einsum("vj,jrc->vrc", model["lbs_weights"].to(dt), A)                  # (V,3,4)
    verts = torch.einsum("vrc,vc->vr", T[:, :, :3], v_posed) + T[:, :, 3] + translation.reshape(1, 3)
    return verts, v_shaped
