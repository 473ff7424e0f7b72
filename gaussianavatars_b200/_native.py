"""ctypes binding of libgaussianavatars_b200.so (the C ABI of include/gab200_rasterizer.h).

There is NO fallback: if the shared library is missing or fails to load, importing the ops raises.  PyTorch is
used only for device memory (the allocation callbacks hand out torch uint8 tensors), streams and autograd glue.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgaussianavatars_b200.so")

ABI_VERSION = 3
INPUT_ACTIVATED = 0
INPUT_BOUND_RAW = 1
SYNC_EXACT, SYNC_LATE, SYNC_NONE = 0, 1, 2
CTR_NOT_MIN_DEPTH_KEY, CTR_MAX_DEPTH_KEY, CTR_NUM_RENDERED, CTR_NUM_LISTED, CTR_BUCKET_OVERFLOW, CTR_CAPACITY, CTR_SEQ = range(7)
NUM_COUNTERS = 8
TUNE_HEAVY_FWD, TUNE_HEAVY_BWD, TUNE_DEPTH_SORT, TUNE_BWD_VARIANT, TUNE_TILE_SORT, TUNE_NVLS_CTAS = 0, 1, 2, 3, 4, 5

ALLOC_FN = C.CFUNCTYPE(C.c_void_p, C.c_void_p, C.c_size_t)


class ForwardArgs(C.Structure):
    _fields_ = [
        ("abi_version", C.c_uint32), ("input_mode", C.c_int32), ("P", C.c_int32), ("sh_degree", C.c_int32),
        ("sh_coeffs", C.c_int32), ("image_width", C.c_int32), ("image_height", C.c_int32),
        ("tanfovx", C.c_float), ("tanfovy", C.c_float), ("scale_modifier", C.c_float),
        ("prefiltered", C.c_int32), ("debug", C.c_int32), ("need_backward", C.c_int32), ("binning_hint", C.c_int32),
        ("exact_binning", C.c_int32), ("depth_hint_lo", C.c_uint32), ("depth_hint_hi", C.c_uint32),
        ("sync_mode", C.c_int32), ("frame_seq", C.c_uint32), ("counters_host", C.c_void_p),
        ("overflow_flag", C.c_void_p),
        ("bg", C.c_void_p), ("viewmatrix", C.c_void_p), ("projmatrix", C.c_void_p), ("campos", C.c_void_p),
        ("means3D", C.c_void_p), ("opacities", C.c_void_p), ("scales", C.c_void_p), ("rotations", C.c_void_p),
        ("cov3D_precomp", C.c_void_p), ("shs", C.c_void_p), ("sh_dc", C.c_void_p), ("sh_rest", C.c_void_p),
        ("colors_precomp", C.c_void_p),
        ("binding", C.c_void_p), ("num_faces", C.c_int32), ("face_center", C.c_void_p),
        ("face_orien_mat", C.c_void_p), ("face_scaling", C.c_void_p),
        ("out_color", C.c_void_p), ("radii", C.c_void_p), ("visibility", C.c_void_p),
        ("alloc_geom", ALLOC_FN), ("alloc_binning", ALLOC_FN), ("alloc_image", ALLOC_FN), ("alloc_user", C.c_void_p),
    ]


class FrameState(C.Structure):
    _fields_ = [
        ("num_rendered", C.c_int64), ("num_candidates", C.c_int64),
        ("geom_buffer", C.c_void_p), ("binning_buffer", C.c_void_p), ("image_buffer", C.c_void_p),
        ("geom_bytes", C.c_size_t), ("binning_bytes", C.c_size_t), ("image_bytes", C.c_size_t),
        ("sorted_selector", C.c_int32), ("sort_bits", C.c_int32), ("depth_bits", C.c_int32),
        ("depth_prefix", C.c_uint32), ("binning_capacity", C.c_int64),
        ("depth_key_min", C.c_uint32), ("depth_key_max", C.c_uint32), ("depth_sort_path", C.c_int32),
        ("attempts", C.c_int32), ("tile_sort_path", C.c_int32), ("reserved0", C.c_int32),
        ("device_counters", C.c_void_p),
    ]


class BackwardArgs(C.Structure):
    _fields_ = [
        ("abi_version", C.c_uint32), ("fwd", C.POINTER(ForwardArgs)), ("state", C.POINTER(FrameState)),
        ("dL_dout_color", C.c_void_p), ("dL_dmeans3D", C.c_void_p), ("dL_dmeans2D", C.c_void_p),
        ("dL_dopacity", C.c_void_p), ("dL_dcolors", C.c_void_p), ("dL_dshs", C.c_void_p), ("dL_dsh_dc", C.c_void_p),
        ("dL_dsh_rest", C.c_void_p), ("dL_dscales", C.c_void_p), ("dL_drotations", C.c_void_p),
        ("dL_dcov3D", C.c_void_p), ("dL_dface_center", C.c_void_p), ("dL_dface_orien_mat", C.c_void_p),
        ("dL_dface_scaling", C.c_void_p), ("grads_are_multicast", C.c_int32),
        ("face_perm", C.c_void_p), ("face_chunk_face", C.c_void_p), ("face_chunk_start", C.c_void_p),
        ("face_chunk_end", C.c_void_p), ("num_face_chunks", C.c_int32),
    ]


class PhotometricArgs(C.Structure):
    """Mirror of gab200_photometric_args."""
    _fields_ = [
        ("abi_version", C.c_uint32), ("channels", C.c_int32), ("height", C.c_int32), ("width", C.c_int32),
        ("gt_is_u8", C.c_int32), ("lambda_dssim", C.c_float),
        ("image", C.c_void_p), ("gt", C.c_void_p), ("grad", C.c_void_p), ("loss", C.c_void_p), ("scratch", C.c_void_p),
    ]


class AdamSegment(C.Structure):
    """Mirror of gab200_adam_segment."""
    _fields_ = [
        ("param", C.c_void_p), ("grad", C.c_void_p), ("exp_avg", C.c_void_p), ("exp_avg_sq", C.c_void_p),
        ("n", C.c_int64), ("lr", C.c_double),
    ]


class DensifyArgs(C.Structure):
    """Mirror of gab200_densify_args."""
    _fields_ = [
        ("abi_version", C.c_uint32), ("P", C.c_int32), ("num_faces", C.c_int32), ("sh_rest_width", C.c_int32),
        ("grad_threshold", C.c_float), ("min_opacity", C.c_float), ("extent", C.c_float), ("percent_dense", C.c_float),
        ("max_screen_size", C.c_float),
        ("xyz", C.c_void_p), ("rotation", C.c_void_p), ("scaling", C.c_void_p), ("opacity", C.c_void_p),
        ("f_dc", C.c_void_p), ("f_rest", C.c_void_p),
        ("exp_avg", C.c_void_p * 6), ("exp_avg_sq", C.c_void_p * 6),
        ("xyz_gradient_accum", C.c_void_p), ("denom", C.c_void_p),
        ("binding", C.c_void_p), ("binding_counter", C.c_void_p), ("face_scaling", C.c_void_p),
        ("scratch", C.c_void_p), ("totals_host", C.c_void_p),
    ]


class DensifyOut(C.Structure):
    """Mirror of gab200_densify_out."""
    _fields_ = [
        ("P_out", C.c_int32), ("n_child_rows", C.c_int32),
        ("xyz", C.c_void_p), ("rotation", C.c_void_p), ("scaling", C.c_void_p), ("opacity", C.c_void_p),
        ("f_dc", C.c_void_p), ("f_rest", C.c_void_p),
        ("exp_avg", C.c_void_p * 6), ("exp_avg_sq", C.c_void_p * 6),
        ("binding", C.c_void_p), ("binding_counter", C.c_void_p), ("noise", C.c_void_p),
        ("src_scratch", C.c_void_p), ("kind_scratch", C.c_void_p), ("noise_row_scratch", C.c_void_p),
    ]


class RegularizeArgs(C.Structure):
    """Mirror of gab200_regularize_args."""
    _fields_ = [
        ("abi_version", C.c_uint32), ("P", C.c_int32), ("metric_xyz", C.c_int32), ("metric_scale", C.c_int32),
        ("threshold_xyz", C.c_float), ("threshold_scale", C.c_float), ("lambda_xyz", C.c_float), ("lambda_scale", C.c_float),
        ("xyz", C.c_void_p), ("scaling", C.c_void_p), ("radii", C.c_void_p), ("binding", C.c_void_p),
        ("face_scaling", C.c_void_p), ("loss", C.c_void_p), ("sums", C.c_void_p),
        ("grad_xyz", C.c_void_p), ("grad_scaling", C.c_void_p), ("grad_face_scaling", C.c_void_p),
    ]


class FlameArgs(C.Structure):
    """Mirror of gab200_flame_args."""
    _fields_ = [
        ("abi_version", C.c_uint32), ("V", C.c_int32), ("n_shape", C.c_int32), ("n_expr", C.c_int32),
        ("J", C.c_int32), ("T", C.c_int32),
        ("v_template", C.c_void_p), ("shapedirs", C.c_void_p), ("posedirs", C.c_void_p), ("J_regressor", C.c_void_p),
        ("lbs_weights", C.c_void_p), ("parents", C.c_void_p), ("J_template", C.c_void_p), ("J_shapedirs", C.c_void_p),
        ("row", C.c_void_p), ("shape", C.c_void_p), ("expr", C.c_void_p), ("rotation", C.c_void_p), ("neck", C.c_void_p),
        ("jaw", C.c_void_p), ("eyes", C.c_void_p), ("translation", C.c_void_p), ("static_offset", C.c_void_p),
        ("verts", C.c_void_p), ("verts_cano", C.c_void_p), ("workspace", C.c_void_p),
        ("grad_shape", C.c_void_p), ("grad_expr", C.c_void_p), ("grad_rotation", C.c_void_p), ("grad_neck", C.c_void_p),
        ("grad_jaw", C.c_void_p), ("grad_eyes", C.c_void_p), ("grad_translation", C.c_void_p),
        ("grad_static_offset", C.c_void_p),
    ]


ADAM_MAX_SEGMENTS = 8
PHOTOMETRIC_SCRATCH_HEAD = 4

EXPORTED_SYMBOLS = ("gab200_forward", "gab200_backward", "gab200_mark_visible", "gab200_bind_activate",
                    "gab200_export_binning", "gab200_launch_count", "gab200_status_string", "gab200_abi_version",
                    "gab200_stage_timing_enable", "gab200_stage_times", "gab200_face_frame_forward",
                    "gab200_face_frame_backward", "gab200_host_times", "gab200_l1_loss_u8", "gab200_l1_loss_u8_backward",
                    "gab200_photometric_loss", "gab200_adam_step", "gab200_tune", "gab200_counters_ok",
                    "gab200_regularize_forward", "gab200_regularize_backward", "gab200_nvls_allreduce", "gab200_densify_scratch_bytes", "gab200_densify_plan", "gab200_densify_apply",
                    "gab200_flame_workspace_bytes", "gab200_flame_forward", "gab200_flame_backward")

_lib = None
_lock = threading.Lock()


class NativeLibraryError(RuntimeError):
    pass


def lib():
    """Load the CUDA library.  Raises NativeLibraryError (never falls back) when it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise NativeLibraryError(
                f"{LIB_PATH} not found: build it with `python -m gaussianavatars_b200.build` "
                "(or __graft_entry__.build()).  gaussianavatars_b200 has no CPU / eager fallback.")
        try:
            L = C.CDLL(LIB_PATH)
        except OSError as e:  # pragma: no cover
            raise NativeLibraryError(f"cannot load {LIB_PATH}: {e}") from e
        for s in EXPORTED_SYMBOLS:
            if not hasattr(L, s):
                raise NativeLibraryError(f"{LIB_PATH} does not export {s}")
        L.gab200_forward.restype = C.c_int64
        L.gab200_forward.argtypes = [C.POINTER(ForwardArgs), C.POINTER(FrameState), C.c_void_p]
        L.gab200_backward.restype = C.c_int32
        L.gab200_backward.argtypes = [C.POINTER(BackwardArgs), C.c_void_p]
        L.gab200_mark_visible.restype = C.c_int32
        L.gab200_mark_visible.argtypes = [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.gab200_bind_activate.restype = C.c_int32
        L.gab200_bind_activate.argtypes = [C.POINTER(ForwardArgs), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_void_p]
        L.gab200_export_binning.restype = C.c_int32
        L.gab200_export_binning.argtypes = [C.POINTER(ForwardArgs), C.POINTER(FrameState), C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_void_p]
        L.gab200_launch_count.restype = C.c_int64
        L.gab200_tune.restype = C.c_int32
        L.gab200_tune.argtypes = [C.c_int32, C.c_int32]
        L.gab200_nvls_allreduce.restype = C.c_int32
        L.gab200_nvls_allreduce.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p]
        L.gab200_regularize_forward.restype = C.c_int32
        L.gab200_regularize_forward.argtypes = [C.POINTER(RegularizeArgs), C.c_void_p]
        L.gab200_regularize_backward.restype = C.c_int32
        L.gab200_regularize_backward.argtypes = [C.POINTER(RegularizeArgs), C.c_void_p, C.c_void_p]
        L.gab200_densify_scratch_bytes.restype = C.c_size_t
        L.gab200_densify_scratch_bytes.argtypes = [C.c_int32, C.c_int32]
        L.gab200_densify_plan.restype = C.c_int32
        L.gab200_densify_plan.argtypes = [C.POINTER(DensifyArgs), C.c_void_p]
        L.gab200_densify_apply.restype = C.c_int32
        L.gab200_densify_apply.argtypes = [C.POINTER(DensifyArgs), C.POINTER(DensifyOut), C.c_void_p]
        L.gab200_flame_workspace_bytes.restype = C.c_size_t
        L.gab200_flame_workspace_bytes.argtypes = [C.c_int32, C.c_int32, C.c_int32]
        L.gab200_flame_forward.restype = C.c_int32
        L.gab200_flame_forward.argtypes = [C.POINTER(FlameArgs), C.c_void_p]
        L.gab200_flame_backward.restype = C.c_int32
        L.gab200_flame_backward.argtypes = [C.POINTER(FlameArgs), C.c_void_p, C.c_void_p]
        L.gab200_counters_ok.restype = C.c_int32
        L.gab200_counters_ok.argtypes = [C.c_void_p, C.c_uint32]
        L.gab200_l1_loss_u8.restype = C.c_int32
        L.gab200_l1_loss_u8.argtypes = [C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.gab200_l1_loss_u8_backward.restype = C.c_int32
        L.gab200_l1_loss_u8_backward.argtypes = [C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.gab200_photometric_loss.restype = C.c_int32
        L.gab200_photometric_loss.argtypes = [C.POINTER(PhotometricArgs), C.c_void_p]
        L.gab200_adam_step.restype = C.c_int32
        L.gab200_adam_step.argtypes = [C.c_int32, C.POINTER(AdamSegment), C.c_int64, C.c_double, C.c_double,
                                       C.c_double, C.c_void_p]
        L.gab200_host_times.restype = None
        L.gab200_host_times.argtypes = [C.POINTER(C.c_double), C.c_int32]
        L.gab200_face_frame_forward.restype = C.c_int32
        L.gab200_face_frame_forward.argtypes = [C.c_int32, C.c_int32] + [C.c_void_p] * 6
        L.gab200_face_frame_backward.restype = C.c_int32
        L.gab200_face_frame_backward.argtypes = [C.c_int32, C.c_int32] + [C.c_void_p] * 7
        L.gab200_status_string.restype = C.c_char_p
        L.gab200_status_string.argtypes = [C.c_int32]
        L.gab200_abi_version.restype = C.c_uint32
        L.gab200_stage_timing_enable.restype = None
        L.gab200_stage_timing_enable.argtypes = [C.c_int32]
        L.gab200_stage_times.restype = C.c_int32
        L.gab200_stage_times.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_int64), C.c_int32]
        if L.gab200_abi_version() != ABI_VERSION:
            raise NativeLibraryError("ABI version mismatch between _native.py and the shared library")
        _lib = L
    return _lib


def check(status: int, what: str):
    if status < 0:
        msg = lib().gab200_status_string(int(status)).decode()
        raise RuntimeError(f"{what} failed: {msg} (status {status})")
    return status


STAGES = ("preprocess", "scan", "emit_keys", "sort", "tile_ranges", "blend_fwd", "blend_bwd", "preprocess_bwd")


def stage_timing(enable: bool):
    lib().gab200_stage_timing_enable(int(enable))


def stage_times(reset: bool = True):
    """{stage: (total_ms, launches)} since the last reset (synchronises the pending events)."""
    ms = (C.c_double * len(STAGES))()
    n = (C.c_int64 * len(STAGES))()
    check(lib().gab200_stage_times(ms, n, int(reset)), "gab200_stage_times")
    return {s: (ms[i], n[i]) for i, s in enumerate(STAGES)}


def host_times(reset: bool = True):
    """Host-side microseconds inside gab200_forward since the last reset (see the header)."""
    out = (C.c_double * 6)()
    lib().gab200_host_times(out, int(reset))
    n = max(out[5], 1.0)
    keys = ("pre_sync_launch", "wait_N", "binning_alloc", "emit_sort_dispatch", "blend_dispatch")
    return {k: out[i] / n for i, k in enumerate(keys)}


def tune(knob: int, value: int = -1) -> int:
    """Set a tuning knob of the library (include/gab200_rasterizer.h GAB200_TUNE_*); returns the previous value."""
    return int(check(lib().gab200_tune(int(knob), int(value)), "gab200_tune"))


def launch_count() -> int:
    return int(lib().gab200_launch_count())


# ---- scratch allocation: the reference's three resizable byte buffers, as torch uint8 tensors -------------------
class _Scratch(threading.local):
    holder = None   # list receiving the tensors of the forward in flight on this thread
    device = None


_scratch = _Scratch()


def _alloc_cb(user, nbytes):
    t = torch.empty(max(int(nbytes), 1), dtype=torch.uint8, device=_scratch.device)
    _scratch.holder.append(t)
    return t.data_ptr()


ALLOC_CALLBACK = ALLOC_FN(_alloc_cb)  # one C thunk for the whole process (kept alive here)


class _InferencePool:
    """no_grad renders reuse three growing buffers per device instead of allocating per frame."""

    def __init__(self):
        self.bufs = {}

    def get(self, device, slot, nbytes):
        key = (device, slot)
        t = self.bufs.get(key)
        if t is None or t.numel() < nbytes:
            t = torch.empty(int(nbytes * 1.25) + 256, dtype=torch.uint8, device=device)
            self.bufs[key] = t
        return t


_pool = _InferencePool()
_pool_slot = threading.local()


def _alloc_pooled_cb(user, nbytes):
    slot = _pool_slot.next
    _pool_slot.next = slot + 1
    return _pool.get(_scratch.device, slot, max(int(nbytes), 1)).data_ptr()


ALLOC_POOLED_CALLBACK = ALLOC_FN(_alloc_pooled_cb)


def begin_forward(device, need_backward: bool):
    """Returns (callback, holder).  holder keeps the per-call scratch alive for backward (None when pooled)."""
    _scratch.device = device
    if need_backward:
        _scratch.holder = []
        return ALLOC_CALLBACK, _scratch.holder
    _pool_slot.next = 0
    return ALLOC_POOLED_CALLBACK, None


def ptr(t):
    return None if t is None else t.data_ptr()
