"""Regenerates tests/golden/flame_vectors.npz and tests/golden/flame_facts.json from the REAL FlameHead of a
GaussianAvatars checkout (flame_model/flame.py + lbs.py, plain torch), run on the synthetic FLAME-shaped model of
gaussianavatars_b200.synthetic.flame_like_model(SEED) -- the licensed arrays are not needed and the model is not stored
(it is regenerated from its seed wherever the vectors are read).

    python tests/golden/make_golden_flame.py

Rows: the 4 frames of demo_flame_param_sample.npz (real pose / expression magnitudes), an all-zero pose (the 1e-8
path of batch_rodrigues), a tiny-angle pose with mixed signs and a large-angle pose near pi.  Stored: the inputs, the
float64 outputs and gradients (dL/dverts of row i = np.random.RandomState(GOUT_SEED + i).standard_normal((V, 3))), and
per row and quantity the max |float32 - float64| of the reference itself over the whole mesh.  The per-vertex arrays
(verts, verts_cano, the static_offset gradient) are kept at `vertex_index` only -- every teeth vertex plus a seeded
sample of the head, N_SAMPLED in all -- so that the file stays small."""
import inspect
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.abspath(os.path.join(HERE, "..", ".."))
sys.path.insert(0, ROOT)

SEED = 0
GOUT_SEED = 100
N_SAMPLED = 1024
GRAD_KEYS = ("shape", "expr", "rotation", "neck", "jaw", "eyes", "translation", "static_offset")


def reference_head(model, dtype):
    from tests import ref_import

    ref_import.prepare()
    from flame_model.flame import FlameHead

    head = FlameHead.__new__(FlameHead)
    torch.nn.Module.__init__(head)
    head.n_shape_params, head.n_expr_params, head.dtype = model["n_shape"], model["n_expr"], dtype
    for k in ("v_template", "shapedirs", "posedirs", "J_regressor", "lbs_weights"):
        head.register_buffer(k, model[k].to(dtype))
    head.register_buffer("parents", model["parents"].long())
    head.register_buffer("faces", model["faces"], persistent=False)
    return head


def inputs():
    demo = np.load(os.path.join(HERE, "demo_flame_param_sample.npz"))
    rows = []
    for t in range(4):
        rows.append(dict(shape=demo["shape"], expr=demo["expr"][t], rotation=demo["rotation"][t],
                         neck=demo["neck_pose"][t], jaw=demo["jaw_pose"][t], eyes=demo["eyes_pose"][t],
                         translation=demo["translation"][t]))
    z3 = np.zeros(3, np.float32)
    rows.append(dict(rows[0], rotation=z3, neck=z3, jaw=z3, eyes=np.zeros(6, np.float32), translation=z3))
    rows.append(dict(rows[1], rotation=np.array([3e-7, -1e-6, 2e-7], np.float32),
                     neck=np.array([-4e-6, 1e-7, 5e-6], np.float32), jaw=np.array([1e-5, -2e-7, 0.0], np.float32),
                     eyes=np.array([2e-6, -3e-6, 1e-7, -1e-5, 4e-7, 0.0], np.float32)))
    axis = np.array([0.3, -0.8, 0.52])
    axis /= np.linalg.norm(axis)
    rows.append(dict(rows[2], rotation=(axis * (np.pi - 2e-3)).astype(np.float32),
                     neck=np.array([0.9, -1.2, 0.4], np.float32), jaw=np.array([0.6, 0.1, -0.05], np.float32),
                     eyes=np.array([0.5, -0.7, 0.1, -2.5, 1.0, 0.3], np.float32)))
    return rows


def static_offset(model):
    v = model["v_template"].double().numpy()
    rs = np.random.RandomState(SEED + 7)
    w = rs.normal(0, 10.0, size=(3, 3))
    return (3e-3 * np.sin(v @ w + rs.uniform(0, 6.28, size=3))).astype(np.float32)


def run(head, row, so, gout, dtype):
    t = {k: torch.tensor(row[k], dtype=dtype)[None].requires_grad_(True) for k in GRAD_KEYS[:-1]}
    so_t = torch.tensor(so, dtype=dtype)[None].requires_grad_(True)
    verts, cano = head(t["shape"], t["expr"], t["rotation"], t["neck"], t["jaw"], t["eyes"], t["translation"],
                       zero_centered_at_root_node=False, return_landmarks=False, return_verts_cano=True,
                       static_offset=so_t)
    (verts[0] * torch.tensor(gout, dtype=dtype)).sum().backward()
    grads = {k: t[k].grad[0].double().numpy() for k in GRAD_KEYS[:-1]}
    grads["static_offset"] = so_t.grad[0].double().numpy()
    return verts[0].detach().double().numpy(), cano[0].detach().double().numpy(), grads


def main():
    from gaussianavatars_b200.synthetic import flame_like_model

    model = flame_like_model(SEED)
    so = static_offset(model)
    rows = inputs()
    V = model["v_template"].shape[0]
    h64, h32 = reference_head(model, torch.float64), reference_head(model, torch.float32)
    n_teeth = 120
    head_sample = np.random.RandomState(SEED + 11).choice(V - n_teeth, N_SAMPLED - n_teeth, replace=False)
    idx = np.sort(np.concatenate([head_sample, np.arange(V - n_teeth, V)])).astype(np.int32)
    out = {k: [] for k in ("verts", "verts_cano", *("grad_" + g for g in GRAD_KEYS), *("spread_" + g for g in
           ("verts", "verts_cano", *GRAD_KEYS)))}
    for i, row in enumerate(rows):
        gout = np.random.RandomState(GOUT_SEED + i).standard_normal((V, 3))
        v64, c64, g64 = run(h64, row, so, gout, torch.float64)
        v32, c32, g32 = run(h32, row, so, gout, torch.float32)
        out["verts"].append(v64[idx])
        out["verts_cano"].append(c64[idx])
        out["spread_verts"].append(np.abs(v32 - v64).max())
        out["spread_verts_cano"].append(np.abs(c32 - c64).max())
        for g in GRAD_KEYS:
            out["grad_" + g].append(g64[g][idx] if g == "static_offset" else g64[g])
            out["spread_" + g].append(np.abs(g32[g] - g64[g]).max())
    arrays = {k: np.stack(v) for k, v in out.items()}
    for k in ("shape", "expr", "rotation", "neck", "jaw", "eyes", "translation"):
        arrays["in_" + k] = np.stack([r[k] for r in rows]).astype(np.float32)
    arrays["in_static_offset"] = so
    arrays["vertex_index"] = idx
    arrays["model_seed"] = np.array(SEED)
    arrays["gout_seed"] = np.array(GOUT_SEED)
    np.savez_compressed(os.path.join(HERE, "flame_vectors.npz"), **arrays)

    from flame_model.flame import FlameHead

    facts = {"FlameHead.forward": str(inspect.signature(FlameHead.forward)),
             "source": "flame_model/flame.py of GaussianAvatars"}
    with open(os.path.join(HERE, "flame_facts.json"), "w") as f:
        json.dump(facts, f, indent=2)
        f.write("\n")
    print({k: float(np.max(v)) for k, v in arrays.items() if k.startswith("spread_")})


if __name__ == "__main__":
    main()
