"""Synthetic workloads of BASELINE.json's shapes (no dataset / licensed FLAME assets travel to the GPU box).

Cameras restate the reference conventions (they are *inputs* of the path, not part of it):
  - `look_at_camera`   : scene/cameras.py:44-47 + utils/graphics_utils.py:38-71 (W2C^T, (P W2C)^T, centre)
  - `orbit_camera`     : utils/viewer_utils.py:20-70,127-170 as used by fps_benchmark_demo.py:21-33
    (OrbitCamera(W,H,r=1,fovy=20,'opencv'): c2w = diag(1,-1,-1), t = (0,0,r) before orbiting; projection from
    intrinsics with z_sign=+1, znear .01, zfar 10; both matrices transposed before use).
Scenes:
  - `random_splats`    : config 1 of SURVEY.md 8(d) (10k random Gaussians, identity binding)
  - `head_mesh` + `avatar_splats` : a FLAME-sized stand-in (10,144 faces; ellipsoidal "head" 0.2x0.3x0.22 m)
    with a heavy-tailed binding histogram and pre-activation parameter statistics calibrated to
    media/306/point_cloud.ply (SURVEY.md 8d: sigmoid(opacity) mean .46, ~6.6 % of splats below 1/255,
    3-sigma radius median ~13 px @1080p, ~15 tiles per splat, N ~ 1.36 M instances for 89k splats).
All generators are seeded and return CPU float32 torch tensors.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Dict, Optional

import numpy as np
import torch


@dataclass
class SyntheticCamera:
    image_width: int
    image_height: int
    FoVx: float
    FoVy: float
    world_view_transform: torch.Tensor  # (4,4) = W2C^T
    full_proj_transform: torch.Tensor   # (4,4) = (P W2C)^T
    camera_center: torch.Tensor         # (3,)
    timestep: int = 0

    @property
    def tanfovx(self):
        return math.tan(self.FoVx * 0.5)

    @property
    def tanfovy(self):
        return math.tan(self.FoVy * 0.5)

    def to(self, device):
        return SyntheticCamera(self.image_width, self.image_height, self.FoVx, self.FoVy,
                               self.world_view_transform.to(device), self.full_proj_transform.to(device),
                               self.camera_center.to(device), self.timestep)


def _projection_gs(znear, zfar, fovx, fovy):
    """utils/graphics_utils.py:51-71."""
    tx, ty = math.tan(fovx / 2), math.tan(fovy / 2)
    top, right = ty * znear, tx * znear
    P = np.zeros((4, 4), np.float32)
    P[0, 0] = 2.0 * znear / (2 * right)
    P[1, 1] = 2.0 * znear / (2 * top)
    P[3, 2] = 1.0
    P[2, 2] = zfar / (zfar - znear)
    P[2, 3] = -(zfar * znear) / (zfar - znear)
    return P


def look_at_camera(W, H, fovx_deg, fovy_deg, w2c: Optional[np.ndarray] = None, znear=0.01, zfar=100.0):
    w2c = np.eye(4, dtype=np.float32) if w2c is None else np.asarray(w2c, np.float32)
    fovx, fovy = math.radians(fovx_deg), math.radians(fovy_deg)
    wv = torch.tensor(w2c).transpose(0, 1).contiguous()
    proj = torch.tensor(_projection_gs(znear, zfar, fovx, fovy)).transpose(0, 1)
    full = (wv.unsqueeze(0).bmm(proj.unsqueeze(0))).squeeze(0).contiguous()
    center = wv.inverse()[3, :3].contiguous()
    return SyntheticCamera(W, H, fovx, fovy, wv, full, center)


def orbit_camera(W, H, r=1.0, fovy_deg=20.0, azimuth_deg=0.0, elevation_deg=0.0, znear=0.01, zfar=10.0):
    focal = H / (2 * np.tan(np.radians(fovy_deg) / 2))
    fovx_deg = np.degrees(2 * np.arctan(W / (2 * focal)))
    pose = np.eye(4, dtype=np.float32)
    pose[2, 3] += r
    az, el = np.radians(azimuth_deg), np.radians(elevation_deg)
    Ry = np.array([[np.cos(az), 0, np.sin(az)], [0, 1, 0], [-np.sin(az), 0, np.cos(az)]], np.float32)
    Rx = np.array([[1, 0, 0], [0, np.cos(el), -np.sin(el)], [0, np.sin(el), np.cos(el)]], np.float32)
    rot = np.eye(4, dtype=np.float32)
    rot[:3, :3] = Ry @ Rx
    pose = rot @ pose
    pose[:, [1, 2]] *= -1  # opencv convention
    cx, cy = W // 2, H // 2
    proj = np.zeros((4, 4))
    proj[0, 0] = focal * 2 / W
    proj[1, 1] = focal * 2 / H
    proj[0, 2] = (W - 2 * cx) / W
    proj[1, 2] = (H - 2 * cy) / H
    proj[2, 2] = (zfar + znear) / (zfar - znear)
    proj[2, 3] = -2 * zfar * znear / (zfar - znear)
    proj[3, 2] = 1.0
    w2c = np.linalg.inv(pose)
    full = proj @ w2c
    return SyntheticCamera(W, H, float(np.radians(fovx_deg)), float(np.radians(fovy_deg)),
                           torch.tensor(w2c).float().T.contiguous(), torch.tensor(full).float().T.contiguous(),
                           torch.tensor(pose[:3, 3]).float().contiguous())


def random_splats(P=10_000, seed=0, sh_degree=0, max_sh_degree=None) -> Dict[str, torch.Tensor]:
    """Config 1: pre-activation parameters of P random Gaussians in front of an identity-view camera."""
    g = torch.Generator().manual_seed(seed)
    M = ((max_sh_degree if max_sh_degree is not None else sh_degree) + 1) ** 2
    xyz = torch.rand(P, 3, generator=g) * 2 - 1
    xyz[:, 2] = xyz[:, 2] * 2 + 4  # z in [2,6]
    xyz[:, :2] *= 2.0
    scaling = math.log(0.03) + 0.5 * torch.randn(P, 3, generator=g)
    rotation = torch.randn(P, 4, generator=g)
    opacity = 2.0 * torch.randn(P, 1, generator=g)
    f_dc = torch.randn(P, 1, 3, generator=g)
    f_rest = 0.3 * torch.randn(P, M - 1, 3, generator=g)
    return dict(_xyz=xyz, _scaling=scaling, _rotation=rotation, _opacity=opacity, _features_dc=f_dc,
                _features_rest=f_rest)


def head_mesh(n_lat=52, n_lon=98, seed=0):
    """Closed ellipsoidal stand-in for the FLAME head: 2*n_lon*(n_lat-1) = 9,996 + jitter faces ~ FLAME's 10,144.
    Returns verts (V,3) float32 centred at the origin and faces (F,3) int64."""
    g = np.random.default_rng(seed)
    rx, ry, rz = 0.105, 0.16, 0.11
    verts = [(0.0, ry, 0.0)]
    for i in range(1, n_lat):
        th = math.pi * i / n_lat
        for j in range(n_lon):
            ph = 2 * math.pi * j / n_lon
            verts.append((rx * math.sin(th) * math.cos(ph), ry * math.cos(th), rz * math.sin(th) * math.sin(ph)))
    verts.append((0.0, -ry, 0.0))
    verts = np.asarray(verts, np.float32)
    verts[1:-1] += g.normal(0, 2e-4, size=(len(verts) - 2, 3)).astype(np.float32)
    faces = []
    for j in range(n_lon):
        faces.append((0, 1 + (j + 1) % n_lon, 1 + j))
    for i in range(n_lat - 2):
        a, b = 1 + i * n_lon, 1 + (i + 1) * n_lon
        for j in range(n_lon):
            jn = (j + 1) % n_lon
            faces.append((a + j, a + jn, b + j))
            faces.append((a + jn, b + jn, b + j))
    last = len(verts) - 1
    a = 1 + (n_lat - 2) * n_lon
    for j in range(n_lon):
        faces.append((last, a + j, a + (j + 1) % n_lon))
    return torch.tensor(verts), torch.tensor(np.asarray(faces, np.int64))


def pose_mesh(verts: torch.Tensor, timestep: int):
    """Documented synthetic per-timestep motion (the licensed FLAME LBS is unavailable): a small rigid head turn
    plus a jaw-like shear of the lower third."""
    t = float(timestep)
    yaw, pitch = 0.15 * math.sin(0.37 * t), 0.08 * math.sin(0.23 * t + 1.0)
    Ry = torch.tensor([[math.cos(yaw), 0, math.sin(yaw)], [0, 1, 0], [-math.sin(yaw), 0, math.cos(yaw)]])
    Rx = torch.tensor([[1, 0, 0], [0, math.cos(pitch), -math.sin(pitch)], [0, math.sin(pitch), math.cos(pitch)]])
    v = verts @ (Ry @ Rx).T.to(verts)
    jaw = torch.clamp((-v[:, 1] - 0.04) / 0.1, 0, 1) * (0.01 * (1 + math.sin(0.5 * t)))
    v = v.clone()
    v[:, 1] -= jaw
    return v


SIZE0, SIZE_SIG = 0.19, 0.85


def avatar_splats(P=100_000, n_faces=10_144, seed=0, sh_degree=3, scale_gain=1.0) -> Dict[str, torch.Tensor]:
    """Bound splats with media/306-like statistics.  `binding` is int32 with a heavy tail (a few faces own
    thousands of splats -- hair/teeth in the real avatar)."""
    g = torch.Generator().manual_seed(seed)
    M = (sh_degree + 1) ** 2
    # heavy-tailed face weights: log-normal + a handful of hot faces
    wts = torch.exp(1.0 * torch.randn(n_faces, generator=g))
    hot = torch.randint(0, n_faces, (12,), generator=g)
    wts[hot] *= 80.0
    binding = torch.multinomial(wts / wts.sum(), P, replacement=True, generator=g).to(torch.int32)
    # every face owns at least one splat for P >= n_faces (the reference never leaves a face empty)
    if P >= n_faces:
        binding[:n_faces] = torch.arange(n_faces, dtype=torch.int32)
    xyz = torch.randn(P, 3, generator=g) * torch.tensor([0.6, 0.6, 0.25])  # local (face) units
    # splat size: clipped log-normal body (radius quantiles of media/306: median 13 px, p90 43, p99 79, max 116 @1080p)
    size = torch.clamp(torch.randn(P, 1, generator=g), -2.5, 1.9)
    jitter = torch.clamp(torch.randn(P, 3, generator=g), -2.0, 2.0)
    scaling = math.log(SIZE0 * scale_gain) + SIZE_SIG * size + 0.35 * jitter
    scaling[:, 2] -= 0.7  # flattened along the face normal
    degenerate = torch.rand(P, generator=g) < 0.003
    scaling[degenerate] = -40.0  # exp -> ~4e-18: the radius-0 / tiny path
    rotation = torch.randn(P, 4, generator=g) * (0.5 + 2.0 * torch.rand(P, 1, generator=g))  # unnormalised raw
    opacity = -0.4 + 3.0 * torch.randn(P, 1, generator=g)
    dead = torch.rand(P, generator=g) < 0.05
    opacity[dead] = -7.0  # sigmoid < 1/255: can never contribute, must keep radii>0
    f_dc = 0.8 * torch.randn(P, 1, 3, generator=g)
    f_rest = 0.08 * torch.randn(P, M - 1, 3, generator=g)
    return dict(_xyz=xyz, _scaling=scaling, _rotation=rotation, _opacity=opacity, _features_dc=f_dc,
                _features_rest=f_rest, binding=binding)


def flame_like_model(seed: int = 0, n_shape: int = 300, n_expr: int = 100, n_lat: int = 52, n_lon: int = 98):
    """A model with FLAME's array shapes and structure, in FlameHead's buffer layout (the licensed arrays are not part of
    this project).  The template is `head_mesh(n_lat, n_lon)` (5000 vertices by default) plus 120 teeth-like vertices
    in 8 rows of 15 that, as FlameHead.add_teeth builds them, have one-hot skinning weights (upper rows on the neck,
    lower rows on the jaw), zero posedirs and J_regressor columns, zero expression directions and shape directions
    copied from the nearest head vertex.  Shape / expression / pose directions are low-frequency in position (posed
    meshes stay smooth), joint regressors are convex averages of nearby vertices, skinning weights are geometric and
    sum to 1.  Joints: 0 global, 1 neck, 2 jaw, 3 / 4 eyes; parents [-1, 0, 1, 1, 1].  Everything is drawn from
    np.random.RandomState(seed), whose stream numpy keeps fixed across versions.  Returns a dict of CPU tensors plus
    n_shape / n_expr."""
    rs = np.random.RandomState(seed)
    head, faces = head_mesh(n_lat, n_lon)
    head = head.numpy().astype(np.float64)
    Vh = head.shape[0]
    # teeth: rows in add_teeth's order (upper root, lower root, upper edge, lower edge, upper root back, upper edge
    # back, lower root back, lower edge back)
    x = np.linspace(-0.03, 0.03, 15)
    row_yz = [(-0.045, 0.085), (-0.095, 0.082), (-0.062, 0.088), (-0.078, 0.084),
              (-0.045, 0.075), (-0.062, 0.078), (-0.095, 0.072), (-0.078, 0.074)]
    teeth = np.concatenate([np.stack([x, np.full(15, y), np.full(15, z)], 1) for y, z in row_yz])
    upper = np.concatenate([np.arange(15 * r, 15 * r + 15) for r in (0, 2, 4, 5)])
    lower = np.concatenate([np.arange(15 * r, 15 * r + 15) for r in (1, 3, 6, 7)])
    v = np.concatenate([head, teeth])
    V, NB = v.shape[0], n_shape + n_expr
    tf = []
    for r0, r1 in ((0, 2), (1, 3), (4, 5), (6, 7)):   # a strip of 28 triangles between two rows
        for i in range(14):
            a, b, c, d = 15 * r0 + i, 15 * r0 + i + 1, 15 * r1 + i, 15 * r1 + i + 1
            tf += [(a, c, b), (b, c, d)]
    faces = torch.cat([faces, torch.tensor(np.asarray(tf, np.int64) + Vh)])

    def smooth(n_fields, amp):   # (V, 3, n_fields): a * sin(w . x + phi), |w| up to ~2 cycles per head
        w = rs.normal(0.0, 12.0, size=(n_fields, 3))
        phi = rs.uniform(0, 2 * np.pi, size=(n_fields, 3))
        a = rs.normal(0.0, 1.0, size=(n_fields, 3)) * amp[:, None]
        arg = head @ w.T                                   # (Vh, n_fields)
        return a.T[None] * np.sin(arg[:, None, :] + phi.T[None])

    decay = lambda n, s: s / (1.0 + np.arange(n) / 30.0)  # noqa: E731
    sd = np.concatenate([smooth(n_shape, decay(n_shape, 2e-3)), smooth(n_expr, decay(n_expr, 1.5e-3))], axis=2)
    nearest = np.argmin(((teeth[:, None, :] - head[None]) ** 2).sum(-1), axis=1)
    sd_teeth = np.zeros((120, 3, NB))
    sd_teeth[:, :, :n_shape] = sd[nearest, :, :n_shape]
    shapedirs = np.concatenate([sd, sd_teeth])
    pd = smooth(36, np.full(36, 4e-3))                     # (Vh, 3, 36)
    posedirs = np.concatenate([pd, np.zeros((120, 3, 36))]).reshape(3 * V, 36).T.copy()
    centres = np.array([[0.0, -0.02, 0.0], [0.0, -0.14, -0.01], [0.0, -0.07, 0.05],
                        [0.035, 0.03, 0.09], [-0.035, 0.03, 0.09]])
    J_regressor = np.zeros((5, V))
    for j, c in enumerate(centres):
        near = np.argsort(((head - c) ** 2).sum(-1))[:24]
        wts = rs.uniform(0.5, 1.5, size=24)
        J_regressor[j, near] = wts / wts.sum()
    sig = np.array([0.25, 0.07, 0.05, 0.02, 0.02])
    d2 = ((head[:, None, :] - centres[None]) ** 2).sum(-1)
    w = np.exp(-d2 / sig ** 2) * np.array([0.2, 1.0, 1.0, 1.0, 1.0])
    w = w / w.sum(1, keepdims=True)
    wt = np.zeros((120, 5))
    wt[upper, 1] = 1.0
    wt[lower, 2] = 1.0
    lbs_weights = np.concatenate([w, wt])
    f32 = lambda a: torch.tensor(np.asarray(a, np.float32))  # noqa: E731
    return dict(v_template=f32(v), shapedirs=f32(shapedirs), posedirs=f32(posedirs), J_regressor=f32(J_regressor),
                parents=torch.tensor([-1, 0, 1, 1, 1], dtype=torch.int64), lbs_weights=f32(lbs_weights), faces=faces,
                n_shape=n_shape, n_expr=n_expr)
