"""Faster R-CNN single-level heads with the reference's interface
(FasterRCNN/building_blocks/proposals.py:373-520 and fastrcnn.py:22-70)."""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _lib

RPN_FEATURE_STRIDE = 16   # FasterRCNN/config.py


def get_anchors():
    """proposals.py:180-196: the 9 ZF-net base anchors (x1, y1, x2, y2)."""
    return np.array([[-84., -40., 99., 55.], [-176., -88., 191., 103.], [-360., -184., 375., 199.],
                     [-56., -56., 71., 71.], [-120., -120., 135., 135.], [-248., -248., 263., 263.],
                     [-36., -80., 51., 95.], [-80., -168., 95., 183.], [-168., -344., 183., 359.]])


class Proposals():
    """``Proposals(mode, rpn_box_class_prob, rpn_bbox)`` (proposals.py:374): numpy/torch inputs of shape
    [B,h,w,18] and [B,h,w,36] -> ``get_proposals()`` [n,5] float32 rows (b, x1, y1, x2, y2): the kept boxes of image 0,
    then those of image 1, and so on, ready for ``roi_pool`` on a [B,h',w',D] feature map. ``num_proposals`` [B] int32
    holds the rows of each image and ``proposals_padded`` [B*post_nms_top_n,5] the same rows followed by zeros.
    Every image is processed as in a batch of one, with one image shape and one set of thresholds for the batch.

    ``image_shape`` / thresholds default to the reference's hard-coded values (proposals.py:378-389) and can be
    overridden for other configurations (e.g. 600x1000, 12000 -> 2000, thr 0.7).
    The top-N ranks the flattened scores (the reference's argsort over an [n,1] array is a bug, see DESIGN.md).
    """

    def __init__(self, mode, rpn_box_class_prob, rpn_bbox, image_shape=(224, 224, 3), nms_threshold=0.2,
                 pre_nms_top_n=None, post_nms_top_n=None, min_box_hw=16):
        self.rpn_box_class_prob = rpn_box_class_prob
        self.rpn_bbox = rpn_bbox
        if mode == 'train':
            self.PRE_NMS_TOP_N, self.POST_NMS_TOP_N = 12000, 2000
        else:
            self.PRE_NMS_TOP_N, self.POST_NMS_TOP_N = 6000, 300
        if pre_nms_top_n is not None:
            self.PRE_NMS_TOP_N = int(pre_nms_top_n)
        if post_nms_top_n is not None:
            self.POST_NMS_TOP_N = int(post_nms_top_n)
        self.NMS_THRESHOLD = nms_threshold
        self.MIN_BOX_HW = min_box_hw
        self.IMAGE_SHAPE = list(image_shape)
        self.build()

    def build(self):
        L = _lib.lib()
        probs, bbox = self.rpn_box_class_prob, self.rpn_bbox
        dt = torch.float64 if (getattr(probs, "dtype", None) in (np.float64, torch.float64)) else torch.float32
        probs = _lib.as_cuda(probs, dt)
        dev = probs.device
        bbox = _lib.as_cuda(bbox, dt, dev)
        base = get_anchors()
        p = _lib.FrcnnParams()
        p.feat_stride, p.image_h, p.image_w = RPN_FEATURE_STRIDE, int(self.IMAGE_SHAPE[0]), int(self.IMAGE_SHAPE[1])
        p.min_box_hw, p.pre_nms_top_n, p.post_nms_top_n = int(self.MIN_BOX_HW), self.PRE_NMS_TOP_N, self.POST_NMS_TOP_N
        p.nms_threshold, p.num_anchors = float(self.NMS_THRESHOLD), base.shape[0]
        for i, v in enumerate(base.reshape(-1)):
            p.base_anchors[i] = float(v)
        B = probs.shape[0]
        out = torch.empty((B * self.POST_NMS_TOP_N, 5), dtype=torch.float32, device=dev)
        num = torch.empty((B,), dtype=torch.int32, device=dev)
        ws = _lib.workspace(L.od_frcnn_proposal_workspace_bytes_batch(B, probs.shape[1], probs.shape[2], ctypes.byref(p)),
                            dev)
        dl = _lib.DL()
        _lib.check(L.od_frcnn_proposal_forward(dl(probs), dl(bbox), ctypes.byref(p), dl(out), dl(num), ws.data_ptr(),
                                               ws.numel(), _lib.stream_ptr(dev)), "od_frcnn_proposal_forward")
        self.proposals_padded, self.num_proposals = out, num
        self.proposals = out[:int(num.sum().item())]   # one host read for the whole batch

    def get_proposals(self):
        return self.proposals


def get_proposal_wrapper(mode, rpn_box_class_prob, rpn_bbox, **kw):
    return Proposals(mode, rpn_box_class_prob, rpn_bbox, **kw).get_proposals()


def roi_pool(feature_map, proposals, image_shape):
    """fastrcnn.py:22-70: crop_and_resize to 14x14 on boxes / (H,W,H,W), then 2x2 max pool -> [n,7,7,D]."""
    fm = _lib.as_cuda(feature_map, torch.float32)
    dev = fm.device
    pr = _lib.as_cuda(proposals, torch.float32, dev)
    out = torch.empty((pr.shape[0], 7, 7, fm.shape[-1]), dtype=torch.float32, device=dev)
    dl = _lib.DL()
    _lib.check(_lib.lib().od_roi_pool_forward(dl(fm), dl(pr), float(image_shape[0]), float(image_shape[1]), dl(out),
                                              _lib.stream_ptr(dev)), "od_roi_pool_forward")
    return out
