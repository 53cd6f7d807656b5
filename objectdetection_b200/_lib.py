"""ctypes binding of ``libodhead.so`` (the C ABI in ``include/odhead.h``).

PyTorch tensors are only the carrier: every tensor crosses the boundary zero-copy as a DLPack
``DLTensor*`` taken from ``torch.utils.dlpack.to_dlpack``.  There is no CPU path: a missing library or a
non-CUDA tensor raises.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_size_t, c_void_p

import torch
from torch.utils.dlpack import to_dlpack

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ODHEAD_LIB") or os.path.join(_HERE, "libodhead.so")   # ODHEAD_LIB: A/B a second build

OD_MAX_LEVELS = 8
OD_MAX_RATIOS = 8


class OdHeadError(RuntimeError):
    """A libodhead.so entry point returned a negative od_status."""

    def __init__(self, status: int, message: str):
        super().__init__(message)
        self.status = status


# ----------------------------------------------------------------------------- C structs
class AnchorSpec(ctypes.Structure):
    _fields_ = [("num_levels", c_int32), ("num_ratios", c_int32),
                ("scales", c_double * OD_MAX_LEVELS), ("ratios", c_double * OD_MAX_RATIOS),
                ("fmap_h", c_int32 * OD_MAX_LEVELS), ("fmap_w", c_int32 * OD_MAX_LEVELS),
                ("fmap_stride", c_int32 * OD_MAX_LEVELS),
                ("anchor_stride", c_int32), ("image_h", c_int32), ("image_w", c_int32)]


class ProposalParams(ctypes.Structure):
    _fields_ = [("bbox_stddev", c_float * 4), ("pre_nms_limit", c_int32), ("post_nms_count", c_int32),
                ("nms_threshold", c_float)]


class ProposalDebug(ctypes.Structure):
    _fields_ = [(n, c_void_p) for n in ("ix", "scores", "bbox_delta", "anchors", "anchor_delta",
                                        "anchor_delta_clipped", "keep_idx", "num_kept")]


class TargetParams(ctypes.Structure):
    _fields_ = [("rois_per_image", c_int32), ("bbox_stddev", c_float * 4), ("mask_h", c_int32), ("mask_w", c_int32),
                ("use_mini_mask", c_int32), ("mask_layout_hwg", c_int32)]


class TargetDebug(ctypes.Structure):
    _fields_ = [(n, c_void_p) for n in ("iou", "roi_iou_max", "pos_indices", "neg_indices", "counts",
                                        "sampled_pos", "sampled_neg", "gt_assignment")]


class RpnTargetParams(ctypes.Structure):
    _fields_ = [("max_rpn_targets", c_int32), ("bbox_stddev", c_double * 4)]


class DetectionParams(ctypes.Structure):
    _fields_ = [("bbox_stddev", c_float * 4), ("min_confidence", c_float), ("nms_threshold", c_float),
                ("max_instances", c_int32)]


class DetectionDebug(ctypes.Structure):
    _fields_ = [(n, c_void_p) for n in ("class_ids", "class_scores", "bbox_delta", "refined_proposals",
                                        "clipped_proposals", "keep_mask", "nms_keep_mask")]


class FrcnnParams(ctypes.Structure):
    _fields_ = [("feat_stride", c_int32), ("image_h", c_int32), ("image_w", c_int32), ("min_box_hw", c_int32),
                ("pre_nms_top_n", c_int32), ("post_nms_top_n", c_int32), ("nms_threshold", c_double),
                ("num_anchors", c_int32), ("base_anchors", c_double * 64)]


# Every symbol include/odhead.h declares, with its ctypes signature (restype, argtypes).
_P = c_void_p
SIGNATURES = {
    "od_version": (c_int, []),
    "od_source_hash": (c_char_p, []),
    "od_strerror": (c_char_p, [c_int]),
    "od_last_error_detail": (c_char_p, []),
    "od_launch_count": (c_int64, []),
    "od_anchor_count": (c_int64, [POINTER(AnchorSpec)]),
    "od_gen_anchors": (c_int, [POINTER(AnchorSpec), c_int, _P, _P]),
    "od_apply_box_deltas": (c_int, [_P, _P, _P, _P]),
    "od_clip_boxes": (c_int, [_P, _P, _P, _P]),
    "od_norm_boxes": (c_int, [_P, c_int32, c_int32, c_int32, _P, _P]),
    "od_topk_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64]),
    "od_topk": (c_int, [_P, c_int64, _P, _P, _P, c_size_t, _P]),
    "od_nms_workspace_bytes": (c_size_t, [c_int64, c_int64]),
    "od_nms": (c_int, [_P, _P, _P, c_float, c_int64, _P, _P, _P, c_size_t, _P]),
    "od_proposal_workspace_bytes": (c_size_t, [c_int64, c_int64, POINTER(ProposalParams)]),
    "od_proposal_forward": (c_int, [_P, _P, _P, POINTER(AnchorSpec), POINTER(ProposalParams), _P,
                                    POINTER(ProposalDebug), _P, c_size_t, _P]),
    "od_proposal_levels_workspace_bytes": (c_size_t, [c_int64, c_int64, POINTER(ProposalParams)]),
    "od_proposal_forward_levels": (c_int, [POINTER(_P), POINTER(_P), c_int32, _P, POINTER(AnchorSpec), POINTER(ProposalParams),
                                           _P, POINTER(ProposalDebug), _P, c_size_t, _P]),
    "od_rpn_loss_workspace_bytes": (c_size_t, [c_int64, c_int64]),
    "od_rpn_loss_forward": (c_int, [_P, _P, _P, _P, _P, _P, _P, _P, c_size_t, _P]),
    "od_mrcnn_loss_forward": (c_int, [_P, _P, _P, _P, _P, _P, _P, _P]),
    "od_pyramid_roi_align_forward": (c_int, [POINTER(_P), c_int32, c_int32, _P, c_int32, c_int32, c_int32, c_int32,
                                             _P, _P, _P]),
    "od_pyramid_roi_align_workspace_bytes": (c_size_t, []),
    "od_pyramid_roi_align_workspace_bytes_n": (c_size_t, [c_int64]),
    "od_pyramid_roi_align_forward_ws": (c_int, [POINTER(_P), c_int32, c_int32, _P, c_int32, c_int32, c_int32, c_int32,
                                                _P, _P, _P, c_size_t, _P]),
    "od_pyramid_roi_align_forward_ordered": (c_int, [POINTER(_P), c_int32, c_int32, _P, c_int32, c_int32, c_int32, c_int32,
                                                     _P, _P, _P, _P, c_size_t, _P]),
    "od_roi_processing_order": (c_int, [_P, c_int32, c_int32, c_int32, c_int32, _P, _P]),
    "od_crop_and_resize": (c_int, [_P, _P, _P, c_int32, c_int32, c_float, _P, _P]),
    "od_detection_target_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64]),
    "od_detection_target_forward": (c_int, [_P, _P, _P, _P, _P, POINTER(TargetParams), _P, _P, _P, _P, _P,
                                            POINTER(TargetDebug), _P, c_size_t, _P]),
    "od_rpn_target_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64]),
    "od_rpn_target_forward": (c_int, [_P, _P, _P, _P, _P, POINTER(RpnTargetParams), _P, _P, _P, _P, _P, c_size_t, _P]),
    "od_detection_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64]),
    "od_detection_forward": (c_int, [_P, _P, _P, _P, POINTER(DetectionParams), _P, POINTER(DetectionDebug), _P,
                                     c_size_t, _P]),
    "od_unmold_detections": (c_int, [_P, _P, _P, _P, _P, _P, _P, _P]),
    "od_frcnn_proposal_workspace_bytes_batch": (c_size_t, [c_int64, c_int64, c_int64, POINTER(FrcnnParams)]),
    "od_frcnn_proposal_workspace_bytes": (c_size_t, [c_int64, c_int64, POINTER(FrcnnParams)]),
    "od_frcnn_proposal_forward": (c_int, [_P, _P, POINTER(FrcnnParams), _P, _P, _P, c_size_t, _P]),
    "od_roi_pool_forward": (c_int, [_P, _P, c_float, c_float, _P, _P]),
}

_lib = None


def lib() -> ctypes.CDLL:
    """Load libodhead.so (built by ``python -m objectdetection_b200.build``). Fails loudly if absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise OdHeadError(-100, f"{LIB_PATH} is missing: the CUDA extension was not built "
                                    "(run `python -m objectdetection_b200.build`); there is no CPU fallback")
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)   # AttributeError if the library does not export a declared symbol
            fn.restype, fn.argtypes = res, args
        # a library older than the sources next to it is refused (it would be tested / benchmarked in their place)
        if os.path.isdir(os.path.join(_HERE, "csrc")) and not os.environ.get("ODHEAD_LIB"):
            from .build import source_hash
            have, want = L.od_source_hash().decode(), source_hash()
            if have != want:
                raise OdHeadError(-100, f"{LIB_PATH} is stale (built from sources {have[:12]}, tree has {want[:12]}): "
                                        "run `python -m objectdetection_b200.build`")
        _lib = L
    return _lib


# ----------------------------------------------------------------------------- DLPack plumbing
_pyapi = ctypes.pythonapi
_pyapi.PyCapsule_GetPointer.restype = c_void_p
_pyapi.PyCapsule_GetPointer.argtypes = [ctypes.py_object, c_char_p]
_pyapi.PyCapsule_IsValid.restype = c_int
_pyapi.PyCapsule_IsValid.argtypes = [ctypes.py_object, c_char_p]


class DL:
    """Holds the DLPack capsules of the tensors of one call and hands out ``DLTensor*`` values.

    A legacy ``"dltensor"`` capsule wraps a ``DLManagedTensor`` whose first member is the ``DLTensor``, so the
    capsule pointer is the ``DLTensor*``.  The capsules stay alive (un-consumed) until this object dies; their
    destructors then release torch's reference.
    """

    def __init__(self):
        self._caps = []

    def __call__(self, t):
        if t is None:
            return None
        if not isinstance(t, torch.Tensor):
            raise TypeError(f"expected a torch.Tensor, got {type(t)}")
        cap = to_dlpack(t)
        if not _pyapi.PyCapsule_IsValid(cap, b"dltensor"):
            raise OdHeadError(-101, "torch did not produce a legacy 'dltensor' capsule")
        self._caps.append(cap)
        return _pyapi.PyCapsule_GetPointer(cap, b"dltensor")


def check(status: int, what: str):
    if status != 0:
        L = lib()
        msg = f"{what}: {L.od_strerror(status).decode()} ({L.od_last_error_detail().decode()})"
        if status in (-2, -3, -5, -8):
            raise ValueError(msg)
        raise OdHeadError(status, msg)


def stream_ptr(device=None) -> int:
    return torch.cuda.current_stream(device).cuda_stream


_workspaces = {}
_retired = []     # superseded workspaces: never freed, a captured CUDA graph may still hold their addresses


def workspace(nbytes: int, device) -> torch.Tensor:
    """A per-(device, stream) scratch buffer that only grows.

    Lifetime rules (CUDA graphs keep raw pointers):
      * a buffer that was ever handed out is never freed: when a call needs more, the old tensor is parked in
        ``_retired`` and stays valid for every graph captured against it;
      * growth is refused DURING stream capture (the new tensor would come from the graph's private pool and then be
        cached for eager use): run the call once eagerly on the capture stream first, as the docstrings say, or
        pre-size with ``reserve_workspace``.
    """
    key = (torch.device(device).index, torch.cuda.current_stream(device).cuda_stream)
    buf = _workspaces.get(key)
    if buf is None or buf.numel() < nbytes:
        if torch.cuda.is_current_stream_capturing():
            raise OdHeadError(-6, f"workspace of {nbytes} bytes would have to be (re)allocated during CUDA graph "
                                  "capture: run the call once eagerly on the capture stream first")
        if buf is not None:
            _retired.append(buf)
        buf = torch.empty(max(int(nbytes), 1 << 20), dtype=torch.uint8, device=device)
        _workspaces[key] = buf
    return buf


_zero_ws = {}


def zeroed_workspace(nbytes: int, device) -> torch.Tensor:
    """A small per-(device, stream) buffer that is zero-initialised once and that the kernels using it leave zeroed
    (od_pyramid_roi_align_forward_ws: the ROI ticket counter). Never freed; allocated outside graph capture."""
    key = (torch.device(device).index, torch.cuda.current_stream(device).cuda_stream)
    buf = _zero_ws.get(key)
    if buf is None or buf.numel() < nbytes:
        if torch.cuda.is_current_stream_capturing():
            raise OdHeadError(-6, "the ROIAlign ticket workspace would have to be allocated during CUDA graph capture: "
                                  "run the call once eagerly on the capture stream first")
        if buf is not None:
            _retired.append(buf)       # a captured graph may still hold its address
        buf = torch.zeros(max(int(nbytes), 256), dtype=torch.uint8, device=device)
        _zero_ws[key] = buf
    return buf


def reserve_workspace(nbytes: int, device) -> None:
    """Pre-size the current stream's workspace (e.g. before capturing a graph with larger shapes)."""
    workspace(nbytes, device)


def as_cuda(x, dtype, device=None) -> torch.Tensor:
    """numpy / host tensor -> CUDA tensor of `dtype` (H2D copy on the current stream); CUDA tensors pass through."""
    if isinstance(x, torch.Tensor):
        t = x
    else:
        import numpy as np
        t = torch.from_numpy(np.ascontiguousarray(x))
    if not t.is_cuda:
        if not torch.cuda.is_available():
            raise OdHeadError(-4, "no CUDA device: objectdetection_b200 has no CPU path")
        if device is None:
            device = torch.device("cuda", torch.cuda.current_device())
        t = t.to(device, non_blocking=True)
    if t.dtype != dtype:
        t = t.to(dtype)
    return t.contiguous()


_const_cache = {}
_CONST_CACHE_MAX = 4096


def const_cuda(arr, dtype, device) -> torch.Tensor:
    """Small host constants (e.g. a normalised window) as CUDA tensors, cached by content, so that repeated calls
    with the same values issue no H2D copy (and the call can be captured in a CUDA graph after one eager run).
    Cached tensors are never evicted (a captured graph may hold their address); past ``_CONST_CACHE_MAX`` distinct
    constants new ones are simply not cached, and a miss during stream capture raises instead of copying."""
    import numpy as np
    a = np.ascontiguousarray(arr)
    key = (torch.device(device).index, str(dtype), a.dtype.str, a.shape, a.tobytes())
    t = _const_cache.get(key)
    if t is None:
        if torch.cuda.is_current_stream_capturing():
            raise OdHeadError(-6, "a host constant (window / image shape) would have to be copied to the device during "
                                  "CUDA graph capture: run the call once eagerly first, or pass a CUDA tensor")
        t = torch.from_numpy(a.copy()).to(device).to(dtype).contiguous()
        if len(_const_cache) < _CONST_CACHE_MAX:
            _const_cache[key] = t
    return t


def make_anchor_spec(image_shape, scales, ratios, feature_map_shapes, feature_map_strides, anchor_stride) -> AnchorSpec:
    s = AnchorSpec()
    if len(scales) > OD_MAX_LEVELS or len(ratios) > OD_MAX_RATIOS:
        raise ValueError("at most 8 pyramid levels and 8 anchor ratios are supported")
    s.num_levels, s.num_ratios = len(scales), len(ratios)
    for i, v in enumerate(scales):
        s.scales[i] = float(v)
        s.fmap_h[i], s.fmap_w[i] = int(feature_map_shapes[i][0]), int(feature_map_shapes[i][1])
        s.fmap_stride[i] = int(feature_map_strides[i])
    for i, v in enumerate(ratios):
        s.ratios[i] = float(v)
    s.anchor_stride, s.image_h, s.image_w = int(anchor_stride), int(image_shape[0]), int(image_shape[1])
    return s
