"""-m gpu: the FLAME kernels (gab200_flame_*) against the reference FlameHead's float64 results, the row-gather
gradients, the drop-in call of FlameGaussianModel.select_mesh_by_timestep, a whole FLAME -> render -> loss step against
the CPU oracles, the graphed step with FLAME inside, and the launch budget."""
import os

import numpy as np
import pytest
import torch

from tests import helpers as h

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "flame_vectors.npz")
GRAD_KEYS = ("shape", "expr", "rotation", "neck", "jaw", "eyes", "translation", "static_offset")
TABLES = {"expr": "expr", "rotation": "rotation", "neck": "neck_pose", "jaw": "jaw_pose", "eyes": "eyes_pose",
          "translation": "translation"}
DEV = torch.device("cuda:0")


class Pipe:
    debug = False
    compute_cov3D_python = False
    convert_SHs_python = False


@pytest.fixture(scope="module")
def golden():
    g = np.load(GOLDEN)
    return {k: g[k] for k in g.files}


@pytest.fixture(scope="module")
def model(golden):
    from gaussianavatars_b200.synthetic import flame_like_model

    return flame_like_model(int(golden["model_seed"]))


@pytest.fixture(scope="module")
def head(model):
    from gaussianavatars_b200 import FusedFlameHead

    return FusedFlameHead(model["v_template"], model["shapedirs"], model["posedirs"], model["J_regressor"],
                          model["parents"], model["lbs_weights"], model["faces"], model["n_shape"],
                          model["n_expr"]).to(DEV)


def _flame_param(golden, rows=(0, 1, 2, 3), requires_grad=True, static=True):
    """flame_param in io.load_flame_param's layout, one frame per golden row."""
    fp = {"shape": torch.tensor(golden["in_shape"][0]),
          "static_offset": torch.tensor(golden["in_static_offset"])[None]}
    for k, key in TABLES.items():
        fp[key] = torch.tensor(golden["in_" + k][list(rows)])
    V = fp["static_offset"].shape[1]
    fp["dynamic_offset"] = torch.zeros(len(rows), V, 3)
    fp = {k: v.to(DEV).contiguous() for k, v in fp.items()}
    for k in TABLES.values():
        fp[k].requires_grad_(requires_grad)
    if static:
        fp["shape"].requires_grad_(requires_grad)
        fp["static_offset"].requires_grad_(requires_grad)
    return fp


def _gate(what, got, ref, spread, floor):
    d = np.abs(got.astype(np.float64) - ref)
    tol = max(4.0 * spread, floor)
    print(f"[flame] {what:<24s} max|d|={d.max():.3e} p50={np.median(d):.3e} p99={np.quantile(d, 0.99):.3e} "
          f"tol={tol:.3e} (4x ref fp32 spread {spread:.3e}, floor {floor:.3e})")
    assert np.isfinite(got).all() and d.max() <= tol, what


@pytest.mark.parametrize("row", range(7))
def test_forward_backward_match_the_reference_flame_head(golden, head, row):
    """Gate: max|d| <= 4x the reference's own fp32-vs-fp64 spread, floor 1e-6 max|v| (vertices) / 1e-4 max|ref|
    (gradients) -- the convention of test_gpu_training.py."""
    ins = {k: torch.tensor(golden["in_" + k][row])[None].to(DEV).requires_grad_(True) for k in GRAD_KEYS[:-1]}
    so = torch.tensor(golden["in_static_offset"])[None].to(DEV).requires_grad_(True)
    verts, cano = head(ins["shape"], ins["expr"], ins["rotation"], ins["neck"], ins["jaw"], ins["eyes"],
                       ins["translation"], zero_centered_at_root_node=False, return_landmarks=False,
                       return_verts_cano=True, static_offset=so)
    assert verts.shape == cano.shape == (1, head.num_verts, 3) and not cano.requires_grad
    gout = np.random.RandomState(int(golden["gout_seed"]) + row).standard_normal((head.num_verts, 3))
    (verts[0] * torch.tensor(gout, dtype=torch.float32, device=DEV)).sum().backward()
    idx = golden["vertex_index"]   # the stored vertices (every teeth vertex + a seeded head sample)
    for name, t in (("verts", verts), ("verts_cano", cano)):
        ref = golden[name][row]
        _gate(name, t[0].detach().cpu().numpy()[idx], ref, float(golden["spread_" + name][row]), 1e-6 * np.abs(ref).max())
    for k in GRAD_KEYS:
        got = so.grad[0].cpu().numpy()[idx] if k == "static_offset" else ins[k].grad[0].cpu().numpy()
        ref = golden["grad_" + k][row]
        _gate("grad_" + k, got, ref, float(golden["spread_" + k][row]), 1e-4 * np.abs(ref).max())


def test_row_gather_accumulates_in_one_row(golden, head):
    V = head.num_verts
    gen = torch.Generator().manual_seed(3)
    g1, g2 = (torch.randn(V, 3, generator=gen).to(DEV) for _ in range(2))

    def grads(fp, pairs):
        loss = sum((head.mesh_at(fp, t) * g).sum() for t, g in pairs)
        loss.backward()
        return {k: v.grad.clone() for k, v in fp.items() if v.grad is not None}

    fp = _flame_param(golden)
    two = grads(fp, [(2, g1), (torch.tensor([2], dtype=torch.int32, device=DEV), g2)])
    one = grads(_flame_param(golden), [(2, g1 + g2)])
    for key in TABLES.values():
        g = two[key]
        assert g.shape == fp[key].shape
        assert torch.count_nonzero(g[[0, 1, 3]]) == 0, f"{key}: rows other than the timestep were written"
        scale = float(one[key].abs().max())
        assert float((g - one[key]).abs().max()) <= 1e-5 * scale, key
    # shape / static_offset not trained: their pointers are NULL and the other gradients do not change
    no_static = grads(_flame_param(golden, static=False), [(1, g1)])
    with_static = grads(_flame_param(golden), [(1, g1)])
    assert "shape" not in no_static and "static_offset" not in no_static
    for key in TABLES.values():
        assert torch.equal(no_static[key], with_static[key]), key


def test_dropin_select_mesh_by_timestep_call_matches_mesh_at(golden, head):
    """The keyword call of FlameGaussianModel.select_mesh_by_timestep (scene/flame_gaussian_model.py:121-134),
    `[[t]]` indexing under autograd included, against mesh_at's row-gather path."""
    gen = torch.Generator().manual_seed(5)
    gout = torch.randn(head.num_verts, 3, generator=gen).to(DEV)
    t = 3
    fp = _flame_param(golden)
    verts, verts_cano = head(
        fp["shape"][None, ...],
        fp["expr"][[t]],
        fp["rotation"][[t]],
        fp["neck_pose"][[t]],
        fp["jaw_pose"][[t]],
        fp["eyes_pose"][[t]],
        fp["translation"][[t]],
        zero_centered_at_root_node=False,
        return_landmarks=False,
        return_verts_cano=True,
        static_offset=fp["static_offset"],
        dynamic_offset=fp["dynamic_offset"][[t]],
    )
    (verts[0] * gout).sum().backward()
    fp2 = _flame_param(golden)
    v2 = head.mesh_at(fp2, t)
    (v2 * gout).sum().backward()
    assert torch.equal(verts[0], v2)
    for k in fp:
        if fp[k].grad is not None:
            assert torch.equal(fp[k].grad, fp2[k].grad), k


def _scene(head, P=15_000, W=400, H=304):
    from gaussianavatars_b200 import synthetic as syn

    params = syn.avatar_splats(P, n_faces=head.faces.shape[0], seed=11, sh_degree=3, scale_gain=2.5)
    cam = syn.orbit_camera(W, H, r=1.0, fovy_deg=20.0, azimuth_deg=15.0)
    return params, cam, W, H


def test_end_to_end_flame_render_loss_gradients(golden, head, model):
    import gaussianavatars_b200 as g
    from gaussianavatars_b200.model import MeshBoundGaussians
    from gaussianavatars_b200.renderer import render
    from oracle.flame import flame_forward
    from oracle.fused_reference import fused_frame

    params, cam, W, H = _scene(head)
    fp = _flame_param(golden)
    pc = MeshBoundGaussians(params, 3, device=DEV, requires_grad=True, flame=head, flame_param=fp)
    t = 2
    pc.select_mesh_by_timestep(t)
    bg = torch.tensor([1.0, 1.0, 1.0])
    out = render(cam.to(DEV), pc, Pipe, bg.to(DEV))
    img = out["render"]
    img.retain_grad()
    gt = torch.randint(0, 256, (3, H, W), generator=torch.Generator().manual_seed(4), dtype=torch.uint8).to(DEV)
    g.l1_loss_u8(img, gt).backward()
    torch.cuda.synchronize()

    # oracle: float64 FLAME (autograd) -> verts -> eager binding + C rasterizer with the same dL/dimage
    m64 = {k: (v.double() if isinstance(v, torch.Tensor) and v.is_floating_point() else v) for k, v in model.items()}
    ins = {k: fp[key].detach().cpu().double()[t].requires_grad_(True) for k, key in TABLES.items()}
    v64, _ = flame_forward(m64, fp["shape"].detach().cpu().double(), ins["expr"], ins["rotation"], ins["neck"],
                           ins["jaw"], ins["eyes"], ins["translation"], fp["static_offset"].detach().cpu().double())
    ref = fused_frame(params, v64.detach().float(), head.faces.cpu(), cam, W, H, bg, 3,
                      dL_dimage=img.grad.detach().cpu())
    v64.backward(torch.tensor(ref["grads"]["verts"], dtype=torch.float64))
    for k, key in TABLES.items():
        got = fp[key].grad[t].cpu().numpy()
        assert torch.count_nonzero(fp[key].grad[[0, 1, 3]]) == 0
        h.assert_grad_tight(got, ins[k].grad.numpy(), what=f"d loss / d {key}")


def test_graphed_frame_with_flame_equals_eager_frames(golden, head):
    import gaussianavatars_b200 as g
    from gaussianavatars_b200.graph import GraphedFrame, camera_block
    from gaussianavatars_b200.model import MeshBoundGaussians
    from gaussianavatars_b200.renderer import render

    params, cam, W, H = _scene(head)
    bg = torch.tensor([1.0, 1.0, 1.0])
    gt = torch.randint(0, 256, (3, H, W), generator=torch.Generator().manual_seed(8), dtype=torch.uint8).to(DEV)

    fp_e = _flame_param(golden, static=False)
    pc_e = MeshBoundGaussians(params, 3, device=DEV, requires_grad=True, flame=head, flame_param=fp_e)
    flame_e = [fp_e[k] for k in TABLES.values()]

    def eager(t):
        for p in pc_e.parameters() + flame_e:
            p.grad = None
        pc_e.select_mesh_by_timestep(t)
        out = render(cam.to(DEV), pc_e, Pipe, bg.to(DEV))
        g.l1_loss_u8(out["render"], gt).backward()
        torch.cuda.synchronize()
        return out["render"].detach().clone(), [p.grad.clone() for p in pc_e.parameters() + flame_e]

    refs = {t: eager(t) for t in (1, 3)}

    fp = _flame_param(golden, static=False)
    pc = MeshBoundGaussians(params, 3, device=DEV, requires_grad=True, flame=head, flame_param=fp)
    fr = GraphedFrame(pc, W, H, cam.FoVx, cam.FoVy, bg, loss="l1_u8", flame=head, flame_param=fp,
                      warm_timesteps=[1, 3])
    with pytest.raises(ValueError, match="timestep="):
        fr.set_inputs(verts=head.v_template)
    fr.set_inputs(camera=camera_block(cam), gt_u8=gt)
    fr.capture()
    for t in (1, 3, 1, 3):
        fr.set_inputs(timestep=t)
        fr.run(check=True)
        torch.cuda.synchronize()
        assert fr.captures == 1
        img, ref_grads = refs[t]
        assert torch.equal(fr.image, img), f"graph replay image differs from the eager frame at timestep {t}"
        got = [p.grad for p in pc.parameters()] + [fp[k].grad for k in TABLES.values()]
        for x, y in zip(got, ref_grads):   # _grads_close of test_gpu_sync_modes.py
            scale = float(y.abs().max()) + 1e-30
            assert float((x - y).abs().max()) <= 2e-5 * scale, "gradients differ beyond atomic-order noise"


def test_launch_budget(golden, head):
    from gaussianavatars_b200 import _native as N

    fp = _flame_param(golden)
    g = torch.ones(head.num_verts, 3, device=DEV)
    head.mesh_at(fp, 0)   # warm (allocator, row index cache)
    torch.cuda.synchronize()
    n0 = N.launch_count()
    v = head.mesh_at(fp, 1)
    n1 = N.launch_count()
    v.backward(g)
    n2 = N.launch_count()
    torch.cuda.synchronize()
    print(f"[flame] library launches: forward {n1 - n0}, backward {n2 - n1}")
    assert n1 - n0 <= 2 and n2 - n1 <= 3
