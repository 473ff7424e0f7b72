"""gaussianavatars_b200 -- B200-native (sm_100a) differentiable Gaussian-splat rasterizer with the GaussianAvatars
FLAME mesh binding fused into preprocess.  Drop-in for the `diff_gaussian_rasterization` operator behind
gaussian_renderer.render() (reference: gaussian_renderer/__init__.py:15,37-52,86-94).

Nothing here falls back to CPU or eager PyTorch: the ops raise if libgaussianavatars_b200.so is missing.
"""
from .rasterizer import (GaussianRasterizationSettings, GaussianRasterizer, rasterize_gaussians, rasterize_bound,
                         bind_activate, set_exact_binning, face_frame, l1_loss_u8)
from .renderer import render, render_bound
from .training import photometric_loss, Adam, binding_regularizers
from .io import load_ply, save_ply, load_flame_param, save_flame_param
from .densify import densify_and_prune, densify_arrays
from .flame import FusedFlameHead

__all__ = ["GaussianRasterizationSettings", "GaussianRasterizer", "rasterize_gaussians", "rasterize_bound",
           "bind_activate", "set_exact_binning", "face_frame", "l1_loss_u8", "render", "render_bound",
           "photometric_loss", "Adam", "binding_regularizers", "load_ply", "save_ply", "load_flame_param", "save_flame_param", "densify_and_prune", "densify_arrays",
           "FusedFlameHead"]
