"""ctypes binding of libb200det.so (the C-ABI declared in include/b200det.h).

There is NO fallback: if the library is missing or a kernel launch fails the call
raises.  torch is used only for device memory and the current stream.
"""
import ctypes
import os

import numpy as np
import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200det.so")

MAX_LEVELS = 8
MAX_ANCHORS = 16

c_void_p, c_int, c_ll, c_float, c_size_t, c_ull = (ctypes.c_void_p, ctypes.c_int, ctypes.c_longlong,
                                                   ctypes.c_float, ctypes.c_size_t, ctypes.c_ulonglong)


class Level(ctypes.Structure):
    _fields_ = [("H", c_int), ("W", c_int), ("A", c_int), ("center_lt", c_int), ("stride", c_float),
                ("ws", c_float * MAX_ANCHORS), ("hs", c_float * MAX_ANCHORS), ("offset", c_ll)]


class Pyramid(ctypes.Structure):
    _fields_ = [("num_levels", c_int), ("_pad", c_int), ("total", c_ll), ("lv", Level * MAX_LEVELS)]


class RpnCfg(ctypes.Structure):
    _fields_ = [("pre_nms", c_int), ("post_nms", c_int), ("max_num", c_int), ("score_mode", c_int),
                ("num_cls_channels", c_int), ("nms_thr_f", c_float), ("min_size", c_float),
                ("means", c_float * 4), ("stds", c_float * 4), ("do_nms", c_int), ("records", c_void_p), ("event_after_select", c_void_p)]


class RoiTargetArgs(ctypes.Structure):
    _fields_ = [("labels", c_void_p), ("max_iou", c_void_p), ("out_ld", c_ll), ("gt", c_void_p), ("gt_ld", c_int),
                ("gt_count", c_void_p), ("gt_label", c_void_p), ("pos_iou", c_float), ("neg_iou", c_float),
                ("min_pos_iou", c_float), ("prepend_gt", c_int), ("census", c_void_p), ("pos_list", c_void_p),
                ("pos_cap", c_int), ("chosen", c_void_p), ("n_chosen", c_void_p), ("max_num", c_int), ("pos_num", c_int),
                ("seed", c_ull), ("seed_step", c_void_p), ("tar_box", c_void_p), ("tar_gt", c_void_p),
                ("tar_param", c_void_p), ("tar_label", c_void_p), ("tar_is_gt", c_void_p), ("means", c_float * 4),
                ("stds", c_float * 4)]


class RoiCfg(ctypes.Structure):
    _fields_ = [("num_levels", c_int), ("C", c_int), ("PH", c_int), ("PW", c_int), ("sampling_ratio", c_int),
                ("aligned", c_int), ("layout", c_int), ("finest_scale", c_float), ("H", c_int * MAX_LEVELS),
                ("W", c_int * MAX_LEVELS), ("spatial_scale", c_float * MAX_LEVELS)]


class DenseLevels(ctypes.Structure):
    """b2d_dense_levels: where the class values of a dense head's rows live (per level: first flat index, base pointer,
    image stride, class stride)."""
    _fields_ = [("num_levels", c_int), ("_pad", c_int), ("offset", c_ll * MAX_LEVELS), ("base", c_void_p * MAX_LEVELS),
                ("img_stride", c_ll * MAX_LEVELS), ("class_stride", c_ll * MAX_LEVELS)]


class B200DetError(RuntimeError):
    pass


_lib = None

_P = c_void_p
_SIGS = {
    "b2d_anchor_grid": [_P, _P, _P, c_int, c_int, c_int, c_float, c_int, _P],
    "b2d_inside_anchor_mask": [_P, _P, c_ll, c_float, c_float, c_float, _P],
    "b2d_inside_grid_mask": [_P, c_int, c_int, c_int, c_int, c_int, _P],
    "b2d_calc_iou": [_P, _P, c_ll, _P, c_ll, _P],
    "b2d_elem_iou": [_P, _P, _P, c_ll, _P],
    "b2d_assign_max_iou": [_P, _P, c_ll, _P, c_ll, _P, c_ll, _P, _P, c_float, _P, c_int, _P, c_int, c_float,
                           c_float, c_float, c_int, _P, _P, c_int, _P, c_size_t, _P],
    "b2d_sample_labels": [_P, _P, _P, c_ll, _P, _P, c_ll, _P, _P, c_int, c_int, c_int, c_int, c_ull, _P, _P],
    "b2d_counter_add": [_P, c_ull, _P],
    "b2d_roi_targets_fused": [_P, _P, c_ll, _P, c_ll, _P, c_ll, _P, c_int, _P, _P, c_int, c_float, c_float, c_float,
                              c_int, _P, _P, c_int, _P, _P, c_int, c_int, c_ull, _P, _P, _P, _P, _P, _P, _P, _P, _P],
    "b2d_anchor_loss_fwd": [_P, _P, _P, _P, _P, c_ll, _P, c_int, _P, c_int, c_float, c_float, c_float, _P, _P, c_int, _P,
                            c_size_t, _P],
    "b2d_anchor_loss_bwd": [_P, _P, _P, _P, _P, _P, _P, c_ll, _P, c_int, _P, c_int, c_float, c_float, c_float, _P, _P,
                            c_int, _P],
    "b2d_fcos_targets": [_P, _P, _P, _P, _P, c_int, _P, _P, _P, _P, c_int, _P],
    "b2d_rcnn_detect": [_P, _P, _P, _P, _P, c_ll, _P, c_ll, _P, _P, c_int, c_int, _P, _P, _P, c_float, c_float, c_int,
                        c_int, c_int, c_int, _P, _P, c_size_t, _P],
    "b2d_rcnn_detect_records": [_P, _P, _P, _P, _P, _P, c_ll, _P, c_ll, _P, _P, c_int, c_int, _P, _P, _P, c_float, c_float,
                                c_int, c_int, c_int, c_int, _P, _P, c_size_t, _P],
    "b2d_dense_detect": [_P, _P, _P, _P, _P, c_ll, _P, _P, _P, c_int, c_int, _P, c_ll, _P, c_float, c_int, c_float, c_int,
                         c_int, c_int, c_int, _P, _P, c_size_t, _P, _P],
    "b2d_dense_detect_records": [_P, _P, _P, _P, _P, _P, c_ll, _P, _P, _P, c_int, c_int, _P, c_ll, _P, c_float, c_int, c_float,
                                 c_int, c_int, c_int, c_int, _P, _P, c_size_t, _P, _P],
    "b2d_dense_select": [_P, _P, _P, _P, _P, _P, c_int, c_int, c_int, _P, c_size_t, _P],
    "b2d_gather_head_outputs": [_P, _P, _P, _P, _P, c_int, _P, _P, c_int, c_int, _P],
    "b2d_roi_align_fwd_batched": [_P, _P, _P, c_ll, _P, c_int, _P, _P],
    "b2d_label_census": [_P, _P, c_int, _P, c_ll, _P, c_ll, c_int, _P],
    "b2d_scatter_sampled": [_P, _P, c_ll, c_ll, _P, _P, c_int, c_int, _P],
    "b2d_bbox2param": [_P, _P, _P, c_ll, _P, _P, _P],
    "b2d_param2bbox": [_P, _P, _P, c_ll, _P, _P, c_int, c_float, c_float, _P],
    "b2d_clamp_bbox": [_P, _P, c_ll, c_float, c_float, _P],
    "b2d_encode_targets": [_P, _P, _P, _P, _P, _P, _P, c_int, _P, c_ll, _P, c_ll, _P, _P, c_int, _P, _P, c_int,
                           _P, _P, c_int, _P],
    "b2d_rpn_proposals": [_P, _P, _P, _P, _P, _P, _P, _P, c_int, _P, _P, c_size_t, _P],
    "b2d_rpn_proposals_targets": [_P, _P, _P, _P, _P, _P, _P, _P, c_int, _P, _P, c_size_t, _P, _P],
    "b2d_topk": [_P, _P, _P, c_ll, _P, c_ll, c_int, c_int, _P, c_size_t, _P],
    "b2d_nms": [_P, _P, _P, _P, c_ll, _P, c_ll, c_int, c_float, c_int, c_int, _P, c_size_t, _P],
    "b2d_roi_align_fwd": [_P, _P, _P, c_ll, _P, _P, c_ll, _P, _P],
    "b2d_roi_align_bwd": [_P, _P, _P, c_ll, _P, _P, c_ll, c_int, _P, _P, c_size_t, _P],
    "b2d_roi_levels": [_P, _P, c_ll, c_ll, c_float, c_int, _P],
    "b2d_nchw_to_nhwc": [_P, _P, c_int, c_int, c_int, c_int, _P],
    "b2d_refine_bboxes": [_P, _P, _P, c_ll, _P, c_ll, _P, _P, c_int, _P, _P, _P, c_int, _P, c_int, _P],
    "b2d_refine_bboxes_argmax": [_P, _P, _P, c_ll, _P, c_ll, _P, c_int, _P, c_int, _P, _P, _P, c_int, _P],
    "b2d_atss_assign": [_P, _P, _P, _P, _P, c_int, _P, _P, _P, c_int, c_int, _P, c_size_t, _P],
    "b2d_fcos_decode": [_P, _P, _P, _P, _P, _P, _P, _P, c_int, c_float, c_float, c_float, _P, c_int, _P],
    "b2d_roi_pool_fwd": [_P, _P, _P, c_int, c_int, c_int, c_int, _P, c_ll, _P, c_ll, c_float, c_int, c_int, _P],
    "b2d_multiclass_nms": [_P, _P, _P, _P, _P, c_int, _P, c_ll, c_int, _P, c_float, _P, c_int, c_float, c_int, c_int, _P, _P,
                           c_size_t, _P],
    "b2d_multiclass_candidates": [_P, _P, _P, _P, _P, _P, _P, c_int, _P, c_ll, c_int, _P, c_float, _P, c_int, c_int, _P],
    "b2d_batched_nms_boxes": [_P, _P, _P, c_ll, _P],
    "b2d_scale_rois": [_P, _P, c_ll, c_ll, c_float, _P],
    "b2d_iou_bin_ids": [_P, _P, _P, c_ll, c_int, _P, _P, _P],
    "b2d_sample_iou_balanced": [_P, _P, _P, c_ll, c_int, c_int, c_int, _P, _P, c_ull, _P],
    "b2d_sampled_ce_fwd": [_P, _P, c_ll, c_int, c_int, c_int, _P, c_ll, _P],
    "b2d_sampled_ce_bwd": [_P, _P, _P, c_ll, c_int, c_int, c_int, _P, c_ll, _P],
    "b2d_ga_pack_scores": [_P, c_ll, _P, _P, _P, c_int, _P],
    "b2d_ga_decode": [_P, _P, _P, _P, _P, c_ll, c_int, _P, _P, _P, _P, _P, c_int, _P, _P, c_float, c_float, c_float, _P],
    "b2d_roi_mark_cells": [_P, _P, c_ll, _P, c_int, _P, _P],
    "b2d_fetch_marked_cells": [_P, _P, _P, c_int, _P, _P, _P],
    "b2d_roi_pool_bwd": [_P, _P, _P, c_int, c_int, c_int, c_int, _P, c_ll, _P, c_ll, c_float, c_int, c_int, _P,
                         c_size_t, _P],
}
_SIZE_FNS = {
    "b2d_rpn_proposals_workspace_bytes": [_P, c_int, _P],
    "b2d_rpn_proposals_debug_offset": [_P, c_int, _P],
    "b2d_topk_workspace_bytes": [c_ll, c_int, c_int],
    "b2d_nms_workspace_bytes": [c_ll, c_int],
    "b2d_roi_align_bwd_workspace_bytes": [c_ll, c_int, _P],
    "b2d_atss_workspace_bytes": [_P, c_int],
    "b2d_rcnn_detect_workspace_bytes": [c_int, c_int],
    "b2d_dense_select_workspace_bytes": [_P, c_int, c_int, c_int],
    "b2d_anchor_loss_workspace_bytes": [_P, c_int],
    "b2d_multiclass_nms_workspace_bytes": [c_int],
    "b2d_sampled_ce_workspace_bytes": [],
    "b2d_roi_cell_bitmap_bytes": [c_int, _P],
}
EXPORTS = sorted(list(_SIGS) + list(_SIZE_FNS) + ["b2d_last_error_string", "b2d_version", "b2d_reload_knobs", "b2d_last_launch_count"])


def lib():
    """Load (once) and return the bound library.  Raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise B200DetError(
            "libb200det.so is not built (%s). Run `python __graft_entry__.py build` "
            "(nvcc, sm_100a). There is no CPU or PyTorch fallback." % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    for name, sig in _SIGS.items():
        fn = getattr(L, name)
        fn.argtypes = sig
        fn.restype = c_int
    for name, sig in _SIZE_FNS.items():
        fn = getattr(L, name)
        fn.argtypes = sig
        fn.restype = c_size_t
    L.b2d_last_error_string.restype = ctypes.c_char_p
    L.b2d_version.restype = c_int
    L.b2d_reload_knobs.restype = None
    L.b2d_last_launch_count.restype = c_int
    _lib = L
    return L


def reload_knobs():
    """Re-read the B2D_* development knobs from the environment (the library reads them once, at first use)."""
    lib().b2d_reload_knobs()


def check(rc, what):
    if rc != 0:
        msg = lib().b2d_last_error_string().decode("utf-8", "replace")
        raise B200DetError("%s failed (rc=%d): %s" % (what, rc, msg))


def call(name, *args):
    check(getattr(lib(), name)(*args), name)


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    return c_void_p(t.data_ptr())


def stream():
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise B200DetError("b200det kernels need CUDA tensors (got a %s tensor); there is no CPU fallback"
                               % t.device.type)


def f32c(t):
    """contiguous fp32 view/copy (the reference works in fp32 throughout)."""
    if t.dtype != torch.float32:
        t = t.to(torch.float32)
    return t.contiguous()


def host_f4(v, default):
    a = np.asarray(default if v is None else v, dtype=np.float32).reshape(-1)
    if a.size != 4:
        raise ValueError("expected 4 values, got %r" % (v,))
    return (c_float * 4)(*a.tolist())


def floor_f32(x):
    """Largest fp32 <= the python double x: makes `iou > thr_f` equal torchvision's CPU
    `(double)iou > thr` for every fp32 iou."""
    f = np.float32(x)
    if float(f) > float(x):
        f = np.nextafter(f, np.float32(-np.inf), dtype=np.float32)
    return float(f)


def make_pyramid(levels):
    """levels: list of dict(stride, H, W, ws, hs, center_lt)."""
    if not 1 <= len(levels) <= MAX_LEVELS:
        raise ValueError("1..%d levels supported" % MAX_LEVELS)
    p = Pyramid()
    p.num_levels = len(levels)
    off = 0
    for i, lv in enumerate(levels):
        A = len(lv["ws"])
        if not 1 <= A <= MAX_ANCHORS:
            raise ValueError("1..%d anchors per cell supported" % MAX_ANCHORS)
        L = p.lv[i]
        L.H, L.W, L.A = int(lv["H"]), int(lv["W"]), A
        L.center_lt = int(bool(lv.get("center_lt", False)))
        L.stride = float(lv["stride"])
        for a in range(A):
            L.ws[a] = float(lv["ws"][a])
            L.hs[a] = float(lv["hs"][a])
        L.offset = off
        off += A * L.H * L.W
    p.total = off
    return p
