"""CPU: the REAL reference's optimizer surgery and checkpoint code (scene/gaussian_model.py:334-419, :89, :111) run
against gaussianavatars_b200.Adam -- the claim INTEGRATION.md makes ("densification and checkpoints work unchanged");
that test needs the reference's own code and skips where it is not installed.  No kernel is launched: the surgery only
edits optimizer state.  The signature of the reference's render() is compared with a stored copy
(tests/golden/make_golden_demo.py)."""
import json
import os

import pytest
import torch

from tests import ref_import

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "reference_facts.json")

NAMES = {"xyz": (3,), "f_dc": (1, 3), "f_rest": (15, 3), "opacity": (1,), "scaling": (3,), "rotation": (4,)}
LRS = {"xyz": 1.6e-4, "f_dc": 2.5e-3, "f_rest": 1.25e-4, "opacity": 5e-2, "scaling": 5e-3, "rotation": 1e-3}


def _model(P, opt_cls):
    ref_import.prepare()
    from scene.gaussian_model import GaussianModel           # REAL reference class

    g = torch.Generator().manual_seed(0)
    m = GaussianModel(3)
    attrs = {"xyz": "_xyz", "f_dc": "_features_dc", "f_rest": "_features_rest", "opacity": "_opacity",
             "scaling": "_scaling", "rotation": "_rotation"}
    groups = []
    for name, shape in NAMES.items():
        p = torch.nn.Parameter(torch.randn(P, *shape, generator=g))
        setattr(m, attrs[name], p)
        groups.append({"params": [p], "lr": LRS[name], "name": name})     # scene/gaussian_model.py:213-220
    m.optimizer = opt_cls(groups, lr=0.0, eps=1e-15)
    m.xyz_gradient_accum = torch.zeros(P, 1)
    m.denom = torch.zeros(P, 1)
    m.max_radii2D = torch.zeros(P)
    return m, attrs


def _warm_state_from_torch(m_ours, P):
    """Two real Adam steps on the CPU with torch's optimizer, state handed over through state_dict."""
    m_t, _ = _model(P, torch.optim.Adam)
    for _ in range(2):
        for gr in m_t.optimizer.param_groups:
            gr["params"][0].grad = torch.randn_like(gr["params"][0])
        m_t.optimizer.step()
    m_ours.optimizer.load_state_dict(m_t.optimizer.state_dict())        # scene/gaussian_model.py:111
    return m_t


@pytest.mark.skipif(not ref_import.available(), reason="the reference's own code is not installed here")
def test_reference_densify_prune_and_checkpoint_code_runs_on_our_adam():
    import gaussianavatars_b200 as g

    P = 40
    m, attrs = _model(P, g.Adam)
    m_t = _warm_state_from_torch(m, P)
    opt = m.optimizer
    for gr in opt.param_groups:
        st = opt.state[gr["params"][0]]
        assert int(st["step"]) == 2 and st["exp_avg"].shape == gr["params"][0].shape

    # densification_postfix -> cat_tensors_to_optimizer (scene/gaussian_model.py:400-438): 7 new splats
    new = {k: torch.randn(7, *s) for k, s in NAMES.items()}
    ref_import.on_cpu(m.densification_postfix, new["xyz"], new["f_dc"], new["f_rest"], new["opacity"], new["scaling"],
                      new["rotation"])          # (the stat buffers it re-creates carry a device="cuda" literal)
    assert m._xyz.shape == (P + 7, 3) and m._features_rest.shape == (P + 7, 15, 3)
    for gr in opt.param_groups:
        p = gr["params"][0]
        st = opt.state[p]
        assert p is getattr(m, attrs[gr["name"]])
        assert st["exp_avg"].shape == p.shape and st["exp_avg_sq"].shape == p.shape
        assert float(st["exp_avg"][P:].abs().sum()) == 0.0 and int(st["step"]) == 2   # new rows start cold, step kept

    # _prune_optimizer (scene/gaussian_model.py:349-372) through the model's own bookkeeping
    keep = torch.ones(P + 7, dtype=torch.bool)
    keep[::5] = False
    tensors = m._prune_optimizer(keep)
    n_keep = int(keep.sum())
    assert set(tensors) == set(NAMES) and all(t.shape[0] == n_keep for t in tensors.values())
    for gr in opt.param_groups:
        assert opt.state[gr["params"][0]]["exp_avg_sq"].shape[0] == n_keep

    # reset_opacity -> replace_tensor_to_optimizer (scene/gaussian_model.py:277-280, :334-347)
    m._opacity = tensors["opacity"]
    out = m.replace_tensor_to_optimizer(torch.full((n_keep, 1), -4.6), "opacity")
    st = opt.state[out["opacity"]]
    assert float(st["exp_avg"].abs().sum()) == 0.0 and float(st["exp_avg_sq"].abs().sum()) == 0.0

    # update_learning_rate walks param_groups by name (scene/gaussian_model.py:228-233)
    m.xyz_scheduler_args = lambda it: 1e-6 * it
    assert m.update_learning_rate(7) == pytest.approx(7e-6)
    assert [gr["lr"] for gr in opt.param_groups if gr["name"] == "xyz"] == [pytest.approx(7e-6)]

    # the checkpoint the reference writes (capture(): optimizer.state_dict(), :89) loads into torch's Adam and steps
    sd = opt.state_dict()
    groups = [{"params": [torch.nn.Parameter(gr["params"][0].detach().clone())], "lr": gr["lr"], "name": gr["name"]}
              for gr in opt.param_groups]
    t_opt = torch.optim.Adam(groups, lr=0.0, eps=1e-15)
    t_opt.load_state_dict(sd)
    for gr in t_opt.param_groups:
        gr["params"][0].grad = torch.ones_like(gr["params"][0])
    t_opt.step()
    assert all(int(t_opt.state[gr["params"][0]]["step"]) == 3 for gr in t_opt.param_groups)
    # ... and our optimizer refuses to step CPU tensors instead of silently doing so
    for gr in opt.param_groups:
        gr["params"][0].grad = torch.ones_like(gr["params"][0])
    with pytest.raises(RuntimeError, match="no CPU or eager fallback"):
        opt.step()
    assert m_t.optimizer.state_dict()["param_groups"][0]["name"] == "xyz"


def test_render_keeps_the_reference_signature():
    """`from gaussianavatars_b200 import render` must accept every call the reference makes
    (train.py:79,124,277; render.py:73; fps_benchmark_demo.py:61; local_viewer.py:630): same leading parameters,
    names and defaults as gaussian_renderer.render (gaussian_renderer/__init__.py:19)."""
    import inspect

    import gaussianavatars_b200 as g

    want = json.load(open(GOLDEN))["render_signature"]      # recorded from the REAL gaussian_renderer.render
    have = list(inspect.signature(g.render).parameters.values())
    assert [p.name for p in have[:len(want)]] == [p["name"] for p in want]
    assert [p.default is not inspect.Parameter.empty for p in have[:len(want)]] == [p["has_default"] for p in want]
    assert [p.default for p in have[:len(want)] if p.default is not inspect.Parameter.empty] == \
        [p["default"] for p in want if p["has_default"]]
    assert all(p.default is not inspect.Parameter.empty for p in have[len(want):])   # extras are optional
