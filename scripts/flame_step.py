"""FLAME on the GPU, measured in one run on one card (writes one JSON document, default profiles/r03/flame_step.json):

  1. the fused FLAME forward and forward+backward per call (gab200_flame_*) against the same maths run eagerly in fp32
     torch + autograd (oracle/flame.py, a restatement of FlameHead.forward -- the reference itself does not run here),
     CUDA events over many calls; the eager arm's kernel count from a separate torch.profiler run;
  2. the config-3 graphed training step (150k splats, 16 cameras, photometric + regularisers, Adam) with FLAME forward
     and backward inside the graph next to the existing graph fed posed vertices, alternated in the same run;
  3. config-5 forward-only frames/s (100k splats, 1920x1080) with select_mesh_by_timestep inside the timed region.

The model is synthetic.flame_like_model(0) (FLAME's array shapes: 5120 vertices, 300 + 100 betas, 5 joints); its
27 MB of arrays stay resident in the 126 MB L2 across back-to-back calls, so (1) is a warm-L2 number."""
import argparse
import json
import math
import os
import re
import subprocess
import sys

sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import gaussianavatars_b200 as g  # noqa: E402
from gaussianavatars_b200 import _native as N  # noqa: E402
from gaussianavatars_b200 import synthetic as syn  # noqa: E402
from gaussianavatars_b200.flame import TABLE_KEYS, FusedFlameHead  # noqa: E402
from gaussianavatars_b200.graph import GraphedFrame, camera_block  # noqa: E402
from gaussianavatars_b200.model import MeshBoundGaussians  # noqa: E402
from gaussianavatars_b200.renderer import render  # noqa: E402
from oracle.flame import flame_forward  # noqa: E402

dev = torch.device("cuda:0")


class Pipe:
    debug = False
    compute_cov3D_python = False
    convert_SHs_python = False


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name(dev)


def timed(fn, iters, warm=10):
    for i in range(warm):
        fn(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def flame_params(m, T, seed=0):
    rs = np.random.RandomState(seed)
    V = m["v_template"].shape[0]
    fp = {"shape": 0.5 * rs.standard_normal(m["n_shape"]), "expr": 0.8 * rs.standard_normal((T, m["n_expr"])),
          "rotation": 0.1 * rs.standard_normal((T, 3)), "neck_pose": 0.05 * rs.standard_normal((T, 3)),
          "jaw_pose": 0.03 * np.abs(rs.standard_normal((T, 3))), "eyes_pose": 0.05 * rs.standard_normal((T, 6)),
          "translation": 0.005 * rs.standard_normal((T, 3)), "static_offset": 1e-3 * rs.standard_normal((1, V, 3)),
          "dynamic_offset": np.zeros((T, V, 3))}
    return {k: torch.tensor(v, dtype=torch.float32, device=dev) for k, v in fp.items()}


def algorithmic_bytes(m):
    V, ns, ne = m["v_template"].shape[0], m["n_shape"], m["n_expr"]
    f = 4
    fwd = f * (V * 3 * (ns + ne) + 36 * 3 * V + V * 3 + V * 5 + 5 * V + 15 * (ns + ne) + 3 * V   # model + offset
               + 3 * V * 3)                                                                     # verts, cano, v_posed
    bwd = f * (V * 3 * ne + 36 * 3 * V + V * 5 + 3 * V + 3 * V + 15 * (ns + ne))                # expr columns only
    return {"forward": fwd, "backward_expr_pose_trans": bwd}


def per_call(m, head, T, iters):
    fp = {k: v.clone().requires_grad_(k in TABLE_KEYS) for k, v in flame_params(m, T).items()}
    gout = torch.randn(head.num_verts, 3, generator=torch.Generator().manual_seed(1)).to(dev)
    m32 = {k: (v.to(dev) if isinstance(v, torch.Tensor) and k != "parents" else v) for k, v in m.items()}

    def eager_inputs(i):
        t = i % T
        return [fp["shape"]] + [fp[k][t] for k in TABLE_KEYS] + [fp["static_offset"][0]]

    def fused_fwd(i):
        with torch.no_grad():
            head.mesh_at(fp, i % T)

    def fused_fb(i):
        for k in TABLE_KEYS:
            fp[k].grad = None
        head.mesh_at(fp, i % T).backward(gout)

    def eager_fwd(i):
        with torch.no_grad():
            flame_forward(m32, *eager_inputs(i))

    def eager_fb(i):
        for k in TABLE_KEYS:
            fp[k].grad = None
        flame_forward(m32, *eager_inputs(i))[0].backward(gout)

    res = {}
    for _ in range(2):   # alternate the arms twice; keep each arm's best
        for name, fn in (("fused_forward_ms", fused_fwd), ("eager_forward_ms", eager_fwd),
                         ("fused_fwd_bwd_ms", fused_fb), ("eager_fwd_bwd_ms", eager_fb)):
            ms = timed(fn, iters)
            res[name] = round(min(ms, res.get(name, 1e9)), 5)
    # outputs of the two arms at the timed size
    with torch.no_grad():
        vf = head.mesh_at(fp, 2)
        ve = flame_forward(m32, *eager_inputs(2))[0]
    res["max_abs_diff_verts_fused_vs_eager"] = float((vf - ve).abs().max())
    grads = {}
    for arm, fn in (("fused", fused_fb), ("eager", eager_fb)):
        fn(2)
        grads[arm] = {k: fp[k].grad[2].clone() for k in TABLE_KEYS}
    res["max_rel_diff_grads_fused_vs_eager"] = {
        k: float((grads["fused"][k] - grads["eager"][k]).abs().max() / grads["eager"][k].abs().max()) for k in TABLE_KEYS}
    # launches: the library's counter; the eager arm's CUDA kernels from a profiler run of one call
    n0 = N.launch_count()
    fused_fb(0)
    res["fused_launches_fwd_bwd"] = N.launch_count() - n0
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        eager_fb(0)
        torch.cuda.synchronize()
    res["eager_cuda_kernels_fwd_bwd"] = sum(1 for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA)
    # device time of each library kernel (profiler run of its own, 50 calls)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(50):
            fused_fb(i)
        torch.cuda.synchronize()
    per = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA and "flame" in e.name:
            key = re.search(r"flame_\w+_kernel", e.name).group(0)
            per[key] = per.get(key, 0.0) + e.device_time_total / 50.0
    res["fused_kernel_us_per_call"] = {k: round(v, 2) for k, v in per.items()}
    return res


def config3(m, head, T, iters, P=150_000):
    out = []
    faces = head.faces
    params = syn.avatar_splats(P, n_faces=faces.shape[0], seed=0, sh_degree=3)
    bg = torch.ones(3, device=dev)
    for (W, H) in ((550, 802), (1920, 1080)):
        cams = [syn.orbit_camera(W, H, azimuth_deg=-60 + 120 * (i + .5) / 16, elevation_deg=5 * math.sin(i)) for i in range(16)]
        blocks = [camera_block(c).to(dev) for c in cams]
        gts = [torch.randint(0, 256, (3, H, W), dtype=torch.uint8, device=dev) for _ in range(2)]
        arms = {}
        for arm in ("verts_input", "flame"):
            fp = {k: v.clone().requires_grad_(k in TABLE_KEYS) for k, v in flame_params(m, T).items()}
            pc = MeshBoundGaussians(params, 3, device=dev, requires_grad=True, flame=head, flame_param=fp)
            groups = [{"params": [p], "lr": 1e-4, "name": str(i)} for i, p in enumerate(pc.parameters())]
            if arm == "flame":
                groups += [{"params": [fp[k] for k in ("rotation", "neck_pose", "jaw_pose", "eyes_pose")], "lr": 1e-5,
                            "name": "pose"}, {"params": [fp["translation"]], "lr": 1e-6, "name": "trans"},
                           {"params": [fp["expr"]], "lr": 1e-3, "name": "expr"}]
                fr = GraphedFrame(pc, W, H, cams[0].FoVx, cams[0].FoVy, bg, loss="photometric", lambda_dssim=0.2,
                                  regularizers={}, warm_cameras=blocks, flame=head, flame_param=fp,
                                  warm_timesteps=[0, 5, 10])
                fr.set_inputs(camera=blocks[0], timestep=0, gt_u8=gts[0])
            else:
                with torch.no_grad():   # posed meshes computed ahead, outside the timed step
                    posed = [head.mesh_at(fp, t).contiguous() for t in range(T)]
                fr = GraphedFrame(pc, W, H, cams[0].FoVx, cams[0].FoVy, bg, loss="photometric", lambda_dssim=0.2,
                                  regularizers={}, warm_cameras=blocks)
                fr.set_inputs(camera=blocks[0], verts=posed[0], gt_u8=gts[0])
            opt = g.Adam(groups, lr=0.0, eps=1e-15)
            fr.capture()

            def step(i, fr=fr, opt=opt, arm=arm, posed=(posed if arm == "verts_input" else None)):
                if arm == "flame":
                    fr.set_inputs(camera=blocks[i % 16], timestep=i % T, gt_u8=gts[i % 2])
                else:
                    fr.set_inputs(camera=blocks[i % 16], verts=posed[i % T], gt_u8=gts[i % 2])
                fr.run()
                opt.step()
            arms[arm] = (fr, step)
        res = {"config": "3", "splats": P, "W": W, "H": H, "verts_input_ms_per_step": [], "flame_ms_per_step": []}
        for _ in range(3):   # alternate
            for arm in ("verts_input", "flame"):
                res[arm + "_ms_per_step"].append(round(timed(arms[arm][1], iters), 4))
        res["graph_overflow"] = any(a[0].overflowed() for a in arms.values())
        res["flame_graph_captures"] = arms["flame"][0].captures
        out.append(res)
        del arms
        torch.cuda.empty_cache()
    return out


def config5(m, head, T, iters, P=100_000, W=1920, H=1080):
    fp = flame_params(m, T)
    params = syn.avatar_splats(P, n_faces=head.faces.shape[0], seed=1, sh_degree=3)
    pc = MeshBoundGaussians(params, 3, device=dev, requires_grad=False, flame=head, flame_param=fp)
    cam = syn.orbit_camera(W, H).to(dev)
    bg = torch.ones(3, device=dev)

    def frame(i):
        with torch.no_grad():
            pc.select_mesh_by_timestep(i % T)
            render(cam, pc, Pipe, bg)

    ms = timed(frame, iters)
    return {"config": "5", "splats": P, "W": W, "H": H, "select_mesh_by_timestep_in_timed_region": True,
            "ms_per_frame": round(ms, 4), "frames_per_s": round(1000.0 / ms, 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(__file__), "..", "profiles", "r03", "flame_step.json"))
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--step-iters", type=int, default=48)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("flame_step.py measures on a GPU; none is visible")
    m = syn.flame_like_model(0)
    head = FusedFlameHead(m["v_template"], m["shapedirs"], m["posedirs"], m["J_regressor"], m["parents"],
                          m["lbs_weights"], m["faces"], m["n_shape"], m["n_expr"]).to(dev)
    T = 16
    doc = {"gpu": gpu_info(), "model": {"V": head.num_verts, "n_shape": m["n_shape"], "n_expr": m["n_expr"], "J": 5},
           "l2_state": "warm: the 27 MB of model arrays stay in L2 across back-to-back calls",
           "eager_arm": "oracle/flame.py in fp32 torch + autograd: a restatement of FlameHead.forward, not the reference",
           "algorithmic_bytes": algorithmic_bytes(m)}
    doc["per_call"] = per_call(m, head, T, a.iters)
    doc["config3_graphed_step"] = config3(m, head, T, a.step_iters)
    doc["config5_forward"] = config5(m, head, T, a.step_iters)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(doc, f, indent=1)
        f.write("\n")
    print(json.dumps(doc))


if __name__ == "__main__":
    main()
