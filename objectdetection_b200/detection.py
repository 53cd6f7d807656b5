"""DetectionLayer with the reference's interface (MaskRCNN/building_blocks/detection.py:8-279)."""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _lib
from .proposals import _stddev4
from .utils import norm_boxes


def unmold_detection(original_image_shape, image_shape, detections, image_window):
    """detection.py:8-53 for ONE image's [M,6] detections: trim at the first class_id == 0, map from the normalised
    window back to original-image pixels (``denorm_boxes``), drop zero-area boxes. Same signature and return values as
    the reference - (boxes [n,4] int32, class_ids [n] int32, scores [n] float32) as numpy arrays - computed by the
    device kernel ``od_unmold_detections`` (the numpy restatement lives in ``oracle/`` as the checker)."""
    det = _lib.as_cuda(detections, torch.float32)
    if det.dim() != 2 or det.shape[1] != 6:
        raise ValueError("detections must be [num_detections, 6] for one image")
    boxes, cls, scores, counts = unmold_detections_batch(np.asarray(original_image_shape).reshape(1, -1), image_shape,
                                                         det[None], np.asarray(image_window).reshape(1, 4))
    n = int(counts[0].item())
    return boxes[0, :n].cpu().numpy(), cls[0, :n].cpu().numpy(), scores[0, :n].cpu().numpy()


def unmold_detections_batch(original_image_shapes, image_shape, detections, image_windows):
    """``unmold_detection`` for a whole batch on the device (e.g. right after the multi-GPU all-gather): detections
    [B,M,6] CUDA float32, image_windows [B,4] pixel windows, original_image_shapes [B,2|3] (or one shape for all).
    Returns (boxes [B,M,4] int32, class_ids [B,M] int32, scores [B,M] float32, counts [B] int32); the first
    ``counts[b]`` rows of image b equal the reference function's output, the rest is zero."""
    det = _lib.as_cuda(detections, torch.float32)
    dev = det.device
    B, M = det.shape[0], det.shape[1]
    if isinstance(image_windows, torch.Tensor) and image_windows.is_cuda:
        win_t = norm_boxes(image_windows.reshape(-1, 4), image_shape[:2])               # detection.py:17, on the device
        if win_t.shape[0] == 1 and B > 1:
            win_t = win_t.expand(B, 4).contiguous()
    else:
        win = norm_boxes(np.asarray(image_windows).reshape(-1, 4), image_shape[:2])      # detection.py:17, host, tiny
        if win.shape[0] == 1 and B > 1:
            win = np.repeat(win, B, 0)
        win_t = _lib.const_cuda(np.ascontiguousarray(win, np.float32), torch.float32, dev)
    shp = np.asarray(original_image_shapes, np.int32).reshape(-1, np.asarray(original_image_shapes).shape[-1])[:, :2]
    if shp.shape[0] == 1 and B > 1:
        shp = np.repeat(shp, B, 0)
    shp_t = _lib.const_cuda(np.ascontiguousarray(shp, np.int32), torch.int32, dev)
    boxes = torch.empty((B, M, 4), dtype=torch.int32, device=dev)
    cls = torch.empty((B, M), dtype=torch.int32, device=dev)
    scores = torch.empty((B, M), dtype=torch.float32, device=dev)
    counts = torch.empty((B,), dtype=torch.int32, device=dev)
    dl = _lib.DL()
    _lib.check(_lib.lib().od_unmold_detections(dl(det), dl(win_t), dl(shp_t), dl(boxes), dl(cls), dl(scores), dl(counts),
                                               _lib.stream_ptr(dev)), "od_unmold_detections")
    return boxes, cls, scores, counts


class DetectionLayer():
    """Per-ROI argmax class -> class-specific delta decode -> clip to window -> bg/score filter -> per-class NMS
    -> top-100 -> zero-padded [B,100,6] rows (y1,x1,y2,x2,class_id,score). Signature of detection.py:57.

    ``mrcnn_class_probs`` and ``mrcnn_bbox`` may each be float32 or bfloat16: a bfloat16 CUDA tensor (2-byte aligned
    probabilities, 8-byte aligned boxes) is read as it is, anything else is converted to float32. bfloat16 values are
    widened exactly, so the detections and DEBUG tensors (float32) are bit for bit those of the call on ``t.float()``."""

    def __init__(self, conf, image_shape, num_batches, window, proposals, mrcnn_class_probs, mrcnn_bbox, DEBUG=False):
        self.image_shape = image_shape
        self.num_batches = num_batches
        self.bbox_stddev = conf.BBOX_STD_DEV
        self.detection_post_nms_instances = conf.DETECTION_POST_NMS_INSTANCES
        self.detection_min_thresh = conf.DETECTION_MIN_THRESHOLD
        self.detection_nms_threshold = conf.DETECTION_NMS_THRESHOLD
        self.DEBUG = DEBUG
        # detection.py:66. A CUDA window is normalised on the device (no host synchronisation); a host window with
        # the reference's numpy formula, then cached on the device by value.
        if isinstance(window, torch.Tensor) and window.is_cuda:
            window = norm_boxes(window.reshape(-1, 4), image_shape[:2])
        else:
            window = norm_boxes(np.asarray(window.numpy() if isinstance(window, torch.Tensor) else window), image_shape[:2])
        self.window = window
        self.detections = self.build(window, proposals, mrcnn_class_probs, mrcnn_bbox)

    def build(self, window, proposals, mrcnn_class_probs, mrcnn_bbox):
        L = _lib.lib()
        props = _lib.as_cuda(proposals, torch.float32)
        dev = props.device
        # bfloat16 head outputs are read as they are (see _lib.read_dtype), anything else as float32
        probs = _lib.as_cuda(mrcnn_class_probs, _lib.read_dtype([mrcnn_class_probs], 2), dev)
        bbox = _lib.as_cuda(mrcnn_bbox, _lib.read_dtype([mrcnn_bbox], 8), dev)
        if isinstance(window, torch.Tensor):
            win = _lib.as_cuda(window, torch.float32, dev).reshape(-1, 4)
        else:
            win = _lib.const_cuda(np.asarray(window, np.float32).reshape(-1, 4), torch.float32, dev)
        B, N, C = probs.shape
        if B != self.num_batches:
            raise ValueError(f"num_batches={self.num_batches} but mrcnn_class_probs has batch {B}")
        M = int(self.detection_post_nms_instances)
        params = _lib.DetectionParams(_stddev4(self.bbox_stddev), float(self.detection_min_thresh),
                                      float(self.detection_nms_threshold), M)
        det = torch.empty((B, M, 6), dtype=torch.float32, device=dev)
        dl = _lib.DL()
        dbg = _lib.DetectionDebug()
        if self.DEBUG:
            self.class_ids = torch.empty((B, N), dtype=torch.int32, device=dev)
            self.class_scores = torch.empty((B, N), dtype=torch.float32, device=dev)
            self.bbox_delta = torch.empty((B, N, 4), dtype=torch.float32, device=dev)
            self.refined_proposals = torch.empty((B, N, 4), dtype=torch.float32, device=dev)
            self.clipped_proposals = torch.empty((B, N, 4), dtype=torch.float32, device=dev)
            self.keep_mask = torch.empty((B, N), dtype=torch.int32, device=dev)
            self.nms_keep_mask = torch.empty((B, N), dtype=torch.int32, device=dev)
            dbg.class_ids, dbg.class_scores, dbg.bbox_delta = dl(self.class_ids), dl(self.class_scores), dl(self.bbox_delta)
            dbg.refined_proposals, dbg.clipped_proposals = dl(self.refined_proposals), dl(self.clipped_proposals)
            dbg.keep_mask, dbg.nms_keep_mask = dl(self.keep_mask), dl(self.nms_keep_mask)
        ws = _lib.workspace(L.od_detection_workspace_bytes(B, N, C), dev)
        _lib.check(L.od_detection_forward(dl(props), dl(probs), dl(bbox), dl(win), ctypes.byref(params), dl(det),
                                          ctypes.byref(dbg), ws.data_ptr(), ws.numel(), _lib.stream_ptr(dev)),
                   "od_detection_forward")
        return det

    def get_detections(self):
        return self.detections

    def debug_outputs(self):
        """The 11 items of detection.py:268-279, same order, same shapes and dtypes. ``class_ids``, ``class_scores``,
        ``bbox_delta``, ``refined_proposals`` and the clipped boxes come straight from the kernels; the index plumbing
        of the TF graph (``indices``, ``mesh``, ``ixs``, :119-125) carries no information beyond ``class_ids`` and is
        synthesised here on request; the per-image pre-NMS lists are the rows selected by the kernel's keep mask
        (class > 0 and score > threshold, ascending ROI index like ``set_intersection``)."""
        keep = self.keep_mask.bool()
        B, N = keep.shape
        dev = keep.device
        indices = torch.arange(N, dtype=torch.int32, device=dev).repeat(B, 1)                 # detection.py:120-124
        mesh = torch.arange(B, dtype=torch.int32, device=dev)[:, None].repeat(1, N)           # detection.py:119
        ixs = torch.stack([mesh, indices, self.class_ids], dim=2)                             # detection.py:125
        clipped_list = [self.clipped_proposals[b][None] for b in range(B)]
        pre_cls = [self.class_ids[b][keep[b]] for b in range(B)]
        pre_scores = [self.class_scores[b][keep[b]] for b in range(B)]
        pre_props = [self.clipped_proposals[b][keep[b]] for b in range(B)]
        return (self.class_ids, indices, mesh, ixs, self.class_scores, self.bbox_delta, self.refined_proposals,
                clipped_list, pre_cls, pre_scores, pre_props)
