"""ProposalLayer with the reference's interface (MaskRCNN/building_blocks/proposals_tf.py:23-326).

``Proposals`` keeps the constructor signature, getters and tensor layouts of the reference class; where the
reference built TF graph nodes, this one launches the sm_100a kernels of ``libodhead.so`` eagerly on the current
CUDA stream. Inputs may be CUDA torch tensors (zero-copy) or host numpy arrays (copied H2D on the stream).
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _lib


def _stddev4(v):
    a = np.asarray(v, dtype=np.float32).reshape(4)
    return (ctypes.c_float * 4)(*[float(x) for x in a])


def apply_box_deltas(pre_nms_anchors, bbox_delta) -> torch.Tensor:
    """proposals_tf.py:23-65. [B,K,4] anchors (y1,x1,y2,x2) + [B,K,4] deltas -> [B,K,4] boxes."""
    a = _lib.as_cuda(pre_nms_anchors, torch.float32)
    d = _lib.as_cuda(bbox_delta, torch.float32, a.device)
    out = torch.empty_like(a)
    dl = _lib.DL()
    _lib.check(_lib.lib().od_apply_box_deltas(dl(a), dl(d), dl(out), _lib.stream_ptr(a.device)), "od_apply_box_deltas")
    return out


def clip_boxes_to_01(anchor_delta, window) -> torch.Tensor:
    """proposals_tf.py:67-94. window is [4] (wy1,wx1,wy2,wx2) or [B,4]."""
    b = _lib.as_cuda(anchor_delta, torch.float32)
    w = _lib.as_cuda(window, torch.float32, b.device)
    out = torch.empty_like(b)
    dl = _lib.DL()
    _lib.check(_lib.lib().od_clip_boxes(dl(b), dl(w), dl(out), _lib.stream_ptr(b.device)), "od_clip_boxes")
    return out


class Proposals():
    """RPN outputs -> top-k -> decode -> clip -> per-image NMS -> zero-padded proposals [B,N,4].

    Same arguments as the reference (proposals_tf.py:103-104). If the three inputs are given the layer runs in
    the constructor (like the reference builds its graph there); otherwise call ``run(...)`` — the equivalent of
    feeding the reference's placeholders. ``anchor_spec`` (optional, from ``utils.anchor_spec``) lets the decode
    kernel regenerate anchors from their index instead of reading ``inp_anchors``.

    ``run_levels(class_logits, bbox)`` takes the RPN head's conv outputs per pyramid level instead
    (``[B,H_l,W_l,2a]`` 'rpn_class_raw' and ``[B,H_l,W_l,4a]`` 'rpn_bbox_pred', rpn.py:50-67): the reshape, the 2-way
    softmax and the concatenation over levels of training.py:146-166 happen inside the layer, nothing is concatenated.

    Head outputs may be float32 or bfloat16 (what ``torch.autocast`` gives a conv): bfloat16 CUDA logits (every level
    bfloat16, 4-byte aligned) and deltas (every level, or ``rpn_bbox``, bfloat16 and 8-byte aligned) are read as they
    are, without a float32 copy; anything else is converted to float32. ``rpn_class_probs`` is float32. bfloat16 values
    are widened exactly, so the proposals and DEBUG tensors (all float32) are bit for bit those of the float32 call on
    ``t.float()``. ``get_proposal_graph()`` returns the inputs as the kernels read them.
    """

    def __init__(self, conf, batch_size, rpn_class_probs=None, rpn_bbox=None, inp_anchors=None,
                 training=False, DEBUG=False, anchor_spec=None):
        self.DEBUG = DEBUG
        self.rpn_bbox_stddev = conf.RPN_BBOX_STDDEV
        self.num_box_before_nms = conf.PRE_NMS_ROIS_COUNT
        self.num_boxes_after_nms = conf.POST_NMS_ROIS_TRAINING if training else conf.POST_NMS_ROIS_INFERENCE
        self.iou_threshold = conf.RPN_NMS_THRESHOLD
        self.batch_size = batch_size
        self.anchor_spec = anchor_spec
        self.rpn_class_probs, self.rpn_bbox, self.input_anchors = rpn_class_probs, rpn_bbox, inp_anchors
        self.proposals = None
        self.anchor_delta_clipped = None
        self._params = _lib.ProposalParams(_stddev4(self.rpn_bbox_stddev), int(self.num_box_before_nms),
                                           int(self.num_boxes_after_nms), float(self.iou_threshold))
        if rpn_class_probs is not None and rpn_bbox is not None and (inp_anchors is not None or anchor_spec is not None):
            self.build()

    def run(self, rpn_class_probs, rpn_bbox, input_anchors=None):
        """Feed-dict style execution (inference.py:138-141)."""
        self.rpn_class_probs, self.rpn_bbox, self.input_anchors = rpn_class_probs, rpn_bbox, input_anchors
        self.build()
        return self.proposals

    def run_levels(self, rpn_class_logits_levels, rpn_bbox_levels, input_anchors=None):
        """The layer on the per-level RPN head outputs (rpn.py:50-67 + training.py:146-166 + this class)."""
        if len(rpn_class_logits_levels) != len(rpn_bbox_levels) or not len(rpn_bbox_levels):
            raise ValueError("one class-logit and one bbox tensor per pyramid level expected")
        self.input_anchors = input_anchors if input_anchors is not None else self.input_anchors
        self.build(levels=(list(rpn_class_logits_levels), list(rpn_bbox_levels)))
        return self.proposals

    def build(self, levels=None):
        L = _lib.lib()
        # bfloat16 logits and deltas go to the kernels as they are (one 4-byte (bg, fg) pair, one 8-byte delta row per
        # load); see _lib.read_dtype. The probabilities of run() are float32.
        if levels is None:
            probs = _lib.as_cuda(self.rpn_class_probs, torch.float32)
            dev = probs.device
            bbox = _lib.as_cuda(self.rpn_bbox, _lib.read_dtype([self.rpn_bbox], 8), dev)
            if probs.dim() != 3:
                raise ValueError("rpn_class_probs must be [batch, anchors, 2]")
            B, A = probs.shape[0], probs.shape[1]
        else:
            logits_dt, deltas_dt = _lib.read_dtype(levels[0], 4), _lib.read_dtype(levels[1], 8)
            logits = [_lib.as_cuda(t, logits_dt) for t in levels[0]]
            dev = logits[0].device
            deltas = [_lib.as_cuda(t, deltas_dt, dev) for t in levels[1]]
            if any(t.dim() != 4 for t in logits + deltas):
                raise ValueError("per-level RPN outputs must be [batch, H, W, channels]")
            B = logits[0].shape[0]
            A = sum(t.shape[1] * t.shape[2] * (t.shape[3] // 2) for t in logits)
        anchors = None if self.input_anchors is None else _lib.as_cuda(self.input_anchors, torch.float32, dev)
        if anchors is None and self.anchor_spec is None:
            raise ValueError("Proposals needs inp_anchors or anchor_spec")
        if B != self.batch_size:
            raise ValueError(f"batch_size={self.batch_size} but the RPN outputs have batch {B}")
        K, N = min(int(self.num_box_before_nms), A), int(self.num_boxes_after_nms)
        self.proposals = torch.empty((B, N, 4), dtype=torch.float32, device=dev)
        self.anchor_delta_clipped = torch.empty((B, K, 4), dtype=torch.float32, device=dev)
        dl = _lib.DL()
        dbg = _lib.ProposalDebug()
        dbg.anchor_delta_clipped = dl(self.anchor_delta_clipped)
        if self.DEBUG:
            self.ix = torch.empty((B, K), dtype=torch.int32, device=dev)
            self.scores = torch.empty((B, K), dtype=torch.float32, device=dev)
            self.bbox_delta = torch.empty((B, K, 4), dtype=torch.float32, device=dev)
            self.anchors = torch.empty((B, K, 4), dtype=torch.float32, device=dev)
            self.anchor_delta = torch.empty((B, K, 4), dtype=torch.float32, device=dev)
            self.keep_idx = torch.empty((B, N), dtype=torch.int32, device=dev)
            self.num_kept = torch.empty((B,), dtype=torch.int32, device=dev)
            dbg.ix, dbg.scores, dbg.bbox_delta = dl(self.ix), dl(self.scores), dl(self.bbox_delta)
            dbg.anchors, dbg.anchor_delta = dl(self.anchors), dl(self.anchor_delta)
            dbg.keep_idx, dbg.num_kept = dl(self.keep_idx), dl(self.num_kept)
        spec = ctypes.byref(self.anchor_spec) if (anchors is None) else None
        if levels is None:
            ws = _lib.workspace(L.od_proposal_workspace_bytes(B, A, ctypes.byref(self._params)), dev)
            _lib.check(L.od_proposal_forward(dl(probs), dl(bbox), dl(anchors), spec, ctypes.byref(self._params),
                                             dl(self.proposals), ctypes.byref(dbg), ws.data_ptr(), ws.numel(),
                                             _lib.stream_ptr(dev)), "od_proposal_forward")
            self.rpn_class_probs, self.rpn_bbox = probs, bbox
        else:
            ws = _lib.workspace(L.od_proposal_levels_workspace_bytes(B, A, ctypes.byref(self._params)), dev)
            lp = (ctypes.c_void_p * len(logits))(*[dl(t) for t in logits])
            bp = (ctypes.c_void_p * len(deltas))(*[dl(t) for t in deltas])
            _lib.check(L.od_proposal_forward_levels(lp, bp, len(logits), dl(anchors), spec, ctypes.byref(self._params),
                                                    dl(self.proposals), ctypes.byref(dbg), ws.data_ptr(), ws.numel(),
                                                    _lib.stream_ptr(dev)), "od_proposal_forward_levels")
            self.rpn_class_logits_levels, self.rpn_bbox_levels = logits, deltas
        if self.DEBUG:
            # the reference scrubs NaNs in DEBUG mode (proposals_tf.py:202-209)
            self.proposals = torch.where(torch.isnan(self.proposals), torch.zeros_like(self.proposals), self.proposals)
        if anchors is not None:
            self.input_anchors = anchors

    def get_proposals(self):
        return self.proposals

    def get_proposal_graph(self):
        return dict(rpn_class_probs=self.rpn_class_probs, rpn_bbox=self.rpn_bbox,
                    input_anchors=self.input_anchors, proposals=self.proposals)

    def get_anchors_delta_clipped(self):
        return self.anchor_delta_clipped

    def debug_outputs(self):
        return self.bbox_delta, self.ix, self.scores, self.anchors, self.anchor_delta


# ----------------------------------------------------------------------------- TF-op level entry points
def top_k(scores, k: int):
    """tf.nn.top_k(sorted=True) over the last axis of a 2-D float32 CUDA tensor (any strides).
    Returns (values [B,k], indices [B,k] int32); ties go to the lower index."""
    if not isinstance(scores, torch.Tensor) or not scores.is_cuda:
        scores = _lib.as_cuda(scores, torch.float32)
    if scores.dtype != torch.float32 or scores.dim() != 2:
        raise ValueError("scores must be a 2-D float32 tensor")
    L = _lib.lib()
    B, A = scores.shape
    dev = scores.device
    vals = torch.empty((B, k), dtype=torch.float32, device=dev)
    idx = torch.empty((B, k), dtype=torch.int32, device=dev)
    ws = _lib.workspace(L.od_topk_workspace_bytes(B, A, k), dev)
    dl = _lib.DL()
    _lib.check(L.od_topk(dl(scores), k, dl(vals), dl(idx), ws.data_ptr(), ws.numel(), _lib.stream_ptr(dev)), "od_topk")
    return vals, idx


def non_max_suppression(boxes, scores, max_output_size: int, iou_threshold: float, num_valid=None):
    """tf.image.non_max_suppression, batched: boxes [B,K,4], scores [B,K] -> (keep_idx [B,max_out] int32 padded
    with -1, num_kept [B] int32). A 2-D/1-D (single image) input returns the trimmed 1-D index tensor like TF."""
    single = (torch.as_tensor(boxes).dim() == 2) if not isinstance(boxes, torch.Tensor) else (boxes.dim() == 2)
    b = _lib.as_cuda(boxes, torch.float32)
    dev = b.device
    s = _lib.as_cuda(scores, torch.float32, dev)
    if single:
        b, s = b[None], s[None]
    B, K = s.shape
    keep = torch.empty((B, max_output_size), dtype=torch.int32, device=dev)
    num = torch.empty((B,), dtype=torch.int32, device=dev)
    nv = None if num_valid is None else _lib.as_cuda(num_valid, torch.int32, dev)
    L = _lib.lib()
    ws = _lib.workspace(L.od_nms_workspace_bytes(B, K), dev)
    dl = _lib.DL()
    _lib.check(L.od_nms(dl(b), dl(s), dl(nv), float(iou_threshold), max_output_size, dl(keep), dl(num),
                        ws.data_ptr(), ws.numel(), _lib.stream_ptr(dev)), "od_nms")
    if single:
        return keep[0, :int(num[0].item())]
    return keep, num
