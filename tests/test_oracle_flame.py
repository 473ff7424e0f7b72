"""CPU: oracle/flame.py (the float64 restatement of FLAME the GPU tests compare against) reproduces the reference
FlameHead's outputs and gradients stored in tests/golden/flame_vectors.npz, and its autograd passes gradcheck."""
import os

import numpy as np
import pytest
import torch

from gaussianavatars_b200.synthetic import flame_like_model
from oracle.flame import flame_forward

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "flame_vectors.npz")
GRAD_KEYS = ("shape", "expr", "rotation", "neck", "jaw", "eyes", "translation", "static_offset")


@pytest.fixture(scope="module")
def golden():
    g = np.load(GOLDEN)
    return {k: g[k] for k in g.files}


@pytest.fixture(scope="module")
def model64(golden):
    m = flame_like_model(int(golden["model_seed"]))
    return {k: (v.double() if isinstance(v, torch.Tensor) and v.is_floating_point() else v) for k, v in m.items()}


def _rel(a, b):
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))


@pytest.mark.parametrize("row", range(7))
def test_oracle_matches_reference_flame_head(golden, model64, row):
    ins = {k: torch.tensor(golden["in_" + k][row], dtype=torch.float64).requires_grad_(True)
           for k in GRAD_KEYS[:-1]}
    so = torch.tensor(golden["in_static_offset"], dtype=torch.float64).requires_grad_(True)
    verts, cano = flame_forward(model64, ins["shape"], ins["expr"], ins["rotation"], ins["neck"], ins["jaw"], ins["eyes"],
                                ins["translation"], so)
    idx = golden["vertex_index"]   # the stored vertices (every teeth vertex + a seeded head sample)
    assert _rel(verts.detach().numpy()[idx], golden["verts"][row]) < 1e-12
    assert _rel(cano.detach().numpy()[idx], golden["verts_cano"][row]) < 1e-12
    V = verts.shape[0]
    gout = np.random.RandomState(int(golden["gout_seed"]) + row).standard_normal((V, 3))
    (verts * torch.tensor(gout)).sum().backward()
    for k in GRAD_KEYS:
        got = so.grad.numpy()[idx] if k == "static_offset" else ins[k].grad.numpy()
        assert _rel(got, golden["grad_" + k][row]) < 1e-12, k


def test_oracle_gradcheck_on_a_reduced_model():
    m = flame_like_model(3, n_shape=4, n_expr=3, n_lat=5, n_lon=6)
    m = {k: (v.double() if isinstance(v, torch.Tensor) and v.is_floating_point() else v) for k, v in m.items()}
    V = m["v_template"].shape[0]
    g = torch.Generator().manual_seed(0)
    r = lambda *s, sc=0.3: (sc * torch.randn(*s, generator=g, dtype=torch.float64)).requires_grad_(True)  # noqa: E731
    args = (r(4), r(3), r(3), r(3), r(3), r(6), r(3, sc=0.01), r(V, 3, sc=1e-3))
    assert torch.autograd.gradcheck(lambda *a: flame_forward(m, *a)[0], args, eps=1e-6, atol=1e-7)
