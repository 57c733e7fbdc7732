"""ctypes binding of the libpnr C ABI (include/pnr.h).  Thin by design: it only checks dtype /
device / contiguity and forwards ``tensor.data_ptr()`` plus the current CUDA stream handle.

There is no CPU or PyTorch fallback: if libpnr.so is missing or a call fails, this raises.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path
from typing import Optional

import torch

# PNR_LIB: load a development variant of the library (tools/timeline.py: the -DPNR_TIMELINE build)
_LIB_PATH = Path(os.environ.get("PNR_LIB") or Path(__file__).resolve().parent / "libpnr.so")
_lib: Optional[C.CDLL] = None

PREC = {"bf16x3": 0, "bf16": 1, "fp16x3": 2, "fp16": 3}


class PnrError(RuntimeError):
    pass


class PnrConfig(C.Structure):
    _fields_ = [("D", C.c_int32), ("W", C.c_int32), ("xyz_res", C.c_int32), ("view_res", C.c_int32),
                ("num_classes", C.c_int32), ("num_instances", C.c_int32), ("precision", C.c_int32),
                ("device", C.c_int32)]


class PnrCompositeOut(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in
                ("rgb_map", "depth_map", "acc_map", "disp_map", "weights", "semantic_map",
                 "instance_map", "fixed_semantic_map", "fixed_instance_map")]


class PnrLossArgs(C.Structure):
    _fields_ = [("R", C.c_int64), ("C", C.c_int32), ("sem_is_prob", C.c_int32)] + \
               [(k, C.c_void_p) for k in ("rgb_map", "rgb_map0", "rgb_gt", "depth_map", "depth_gt", "semantic_map",
                                          "fixed_semantic_map", "label", "label_weight")] + \
               [(k, C.c_float) for k in ("w_rgb", "w_depth", "w_sem", "w_fix", "inv_n_rgb", "inv_n_depth", "inv_n_sem", "eps")] + \
               [(k, C.c_void_p) for k in ("per_ray", "d_rgb_map", "d_rgb_map0", "d_depth_map", "d_semantic_map",
                                          "d_fixed_semantic_map")]


class PnrCompositeGrads(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in
                ("rgb_map", "depth_map", "acc_map", "weights", "semantic_map",
                 "instance_map", "fixed_semantic_map", "fixed_instance_map")]


class PnrRenderArgs(C.Structure):
    """pnr_render_args of include/pnr.h (same field order)."""
    _fields_ = [("rays", C.c_void_p), ("R", C.c_int64), ("near", C.c_void_p), ("far", C.c_void_p),
                ("aabb_host", C.POINTER(C.c_float)), ("near_min", C.c_float), ("far_default", C.c_float),
                ("box_center", C.c_void_p), ("box_half", C.c_void_p), ("box_rot", C.c_void_p),
                ("box_sem", C.c_void_p), ("box_inst", C.c_void_p), ("B", C.c_int32), ("M", C.c_int32),
                ("N", C.c_int32), ("Ni", C.c_int32), ("t_vals", C.c_void_p), ("u", C.c_void_p),
                ("perturb", C.c_float), ("u_fine", C.c_void_p), ("u_fine_stride", C.c_int64),
                ("sample_mode", C.c_int32), ("white_bkgd", C.c_int32), ("sem_softmax", C.c_int32),
                ("mask_outside", C.c_int32), ("bound_by_primitives", C.c_int32),
                ("out", PnrCompositeOut), ("out0", PnrCompositeOut), ("z_vals", C.c_void_p), ("z_vals0", C.c_void_p),
                ("hit_mask", C.c_void_p), ("box_id", C.c_void_p), ("t_in", C.c_void_p), ("t_out", C.c_void_p),
                ("sample_box", C.c_void_p), ("near_out", C.c_void_p), ("far_out", C.c_void_p),
                ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t)]


class PnrEvalArgs(C.Structure):
    """pnr_eval_args of include/pnr.h (same field order)."""
    _fields_ = [("R", C.c_int64), ("C", C.c_int32), ("H", C.c_int32), ("W", C.c_int32)] + \
               [(k, C.c_void_p) for k in ("sem_pred", "sem_gt", "pan_pred", "pan_gt", "is_thing")] + \
               [("label_divisor", C.c_int32)] + \
               [(k, C.c_void_p) for k in ("rgb_pred", "rgb_gt", "depth_pred", "depth_gt")] + \
               [("min_depth", C.c_float), ("max_depth", C.c_float), ("stats", C.c_void_p), ("workspace", C.c_void_p),
                ("workspace_bytes", C.c_size_t)]


SAMPLE_MODE = {"uniform": 0, "intervals": 1}
COMM_ID_BYTES = 128

# name -> (restype, argtypes); mirrors include/pnr.h one to one
_vp, _i32, _i64, _f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_float
SIGNATURES = {
    "pnr_version": (C.c_int, []),
    "pnr_last_error": (C.c_char_p, []),
    "pnr_create": (C.c_int, [C.POINTER(PnrConfig), C.POINTER(_vp)]),
    "pnr_destroy": (C.c_int, [_vp]),
    "pnr_status": (C.c_int, [_vp, C.POINTER(C.c_uint32), _i32, _vp]),
    "pnr_load_weights": (C.c_int, [_vp, C.POINTER(_vp), C.POINTER(_i64), _i32]),
    "pnr_intersect": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "pnr_scene_near_far": (C.c_int, [_vp, _i64, C.POINTER(_f32), _f32, _f32, _vp, _vp, _vp]),
    "pnr_bound_by_primitives": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i32, _vp, _vp, _vp]),
    "pnr_sample_stratified": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i32, _f32, _vp, _vp, _vp, _i32, _vp, _vp, _vp]),
    "pnr_sample_intervals": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i32, _f32, _vp, _vp, _vp, _i32, _vp, _vp, _vp]),
    "pnr_tag_samples": (C.c_int, [_vp, _i64, _i32, _vp, _vp, _vp, _i32, _vp, _vp]),
    "pnr_generate_rays": (C.c_int, [_i32, _i32, _i32, _i32, _i32, C.POINTER(_f32), C.POINTER(_f32), _vp, _vp]),
    "pnr_encode": (C.c_int, [_vp, _i64, _i32, _vp, _vp]),
    "pnr_mlp_forward": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, _i32, _vp, _vp]),
    "pnr_mlp_composite": (C.c_int, [_vp, _vp, _vp, _i64, _i32, _i32, _i32, _vp, _vp, _vp, _i32,
                                    C.POINTER(PnrCompositeOut), _vp]),
    "pnr_mlp_forward_timeline": (C.c_int, [_vp, _vp, _vp, _i64, _i32, _vp, _vp, _vp]),
    "pnr_debug_timeline": (C.c_int, [_vp, _vp]),
    "pnr_mlp_backward_trunk": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i32, _vp, C.c_float, _vp, _i32, _vp, _vp, _vp]),
    "pnr_mlp_trunk_forward": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i32, _vp, _vp]),
    "pnr_composite": (C.c_int, [_vp, _vp, _vp, _i64, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _i32,
                                C.POINTER(PnrCompositeOut), _vp]),
    "pnr_losses": (C.c_int, [C.POINTER(PnrLossArgs), _vp]),
    "pnr_panoptic_fuse": (C.c_int, [_vp, _vp, _i64, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "pnr_hashgrid_encode": (C.c_int, [_vp, _i64, _vp, _vp, _i32, _i32, _i32, C.c_float, C.c_float, _vp, _vp]),
    "pnr_hashgrid_backward": (C.c_int, [_vp, _i64, _vp, _vp, _i32, _i32, _i32, C.c_float, C.c_float, _vp, _vp]),
    "pnr_label_tiles": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "pnr_composite_backward": (C.c_int, [_vp, _vp, _vp, _i64, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp,
                                         _i32, C.POINTER(PnrCompositeGrads), _vp, _vp]),
    "pnr_wgrad_workspace_bytes": (C.c_size_t, [_i32, _i32]),
    "pnr_wgrad": (C.c_int, [_vp, _i64, _i32, _vp, _i64, _i32, _i64, _i32, _vp, _vp, _i64, _vp, _i32, _vp, C.c_size_t, _vp]),
    "pnr_linear_workspace_bytes": (C.c_size_t, [_i32, _i32]),
    "pnr_linear": (C.c_int, [_vp, _i64, _i32, _vp, _i64, _i32, _vp, _i32, _i64, _i32, _i32, _vp, _vp, _i64, _vp, C.c_size_t, _vp]),
    "pnr_sample_pdf": (C.c_int, [_vp, _vp, _i64, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "pnr_update_weights": (C.c_int, [_vp, C.POINTER(_vp), _i32, _vp]),
    "pnr_program_host": (C.c_int, [C.POINTER(PnrConfig), C.POINTER(_vp), C.POINTER(_i64), _i32, _i32, _vp, C.c_size_t,
                                   C.POINTER(C.c_size_t), _vp, C.c_size_t, C.POINTER(C.c_size_t), _vp, C.c_size_t,
                                   C.POINTER(C.c_size_t)]),
    "pnr_render_fused": (C.c_int, [_vp, _vp, C.POINTER(PnrRenderArgs), _vp]),
    "pnr_workspace_bytes": (C.c_size_t, [_vp, _i64, _i32, _i32]),
    "pnr_comm_available": (C.c_int, []),
    "pnr_comm_unique_id": (C.c_int, [C.POINTER(C.c_uint8)]),
    "pnr_comm_init": (C.c_int, [C.POINTER(_vp), C.POINTER(C.c_uint8), _i32, _i32, _i32]),
    "pnr_comm_destroy": (C.c_int, [_vp]),
    "pnr_allgather_outputs": (C.c_int, [_vp, _vp, _vp, C.c_size_t, _vp]),
    "pnr_eval_stats_bytes": (C.c_size_t, [_i32]),
    "pnr_eval_workspace_bytes": (C.c_size_t, [_i64, _i32, _i32]),
    "pnr_eval_frame": (C.c_int, [C.POINTER(PnrEvalArgs), _vp]),
    "pnr_launch_count": (_i64, [_i32]),
}


def lib() -> C.CDLL:
    """Load libpnr.so (once).  Fails loudly: the product has no path that works without it."""
    global _lib
    if _lib is None:
        if not _LIB_PATH.exists():
            raise PnrError(f"{_LIB_PATH} is missing - run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(nvcc, sm_100a).  panopticnerf_b200 has no CPU or PyTorch fallback.")
        L = C.CDLL(str(_LIB_PATH))
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)          # AttributeError here = header/library mismatch
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib().pnr_last_error()
        raise PnrError(f"{what or 'libpnr'} failed (rc={rc}): {msg.decode() if msg else '?'}")


def stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def ptr(t: Optional[torch.Tensor], dtype: Optional[torch.dtype] = None, name: str = "tensor"):
    """Device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise PnrError(f"{name}: expected a CUDA tensor, got {t.device} - panopticnerf_b200 is GPU-only "
                       "(no CPU fallback)")
    if dtype is not None and t.dtype != dtype:
        raise PnrError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise PnrError(f"{name}: expected a contiguous tensor")
    return t.data_ptr()
