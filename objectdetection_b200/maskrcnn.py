"""PyramidROIAlign with the reference's interface (MaskRCNN/building_blocks/maskrcnn.py:35-187).

``MaskRCNN`` keeps the reference constructor signature, ``roi_pooling`` and ``get_pooled_rois``; the dense
classifier head (maskrcnn.py:189-315, conv/FC — cuDNN/cuBLAS territory) is outside the detection-head hot path
and is not part of this package.
"""
from __future__ import annotations

import ctypes

import torch

from . import _lib


def roi_processing_order(proposals, image_shape, levels=(2, 3, 4, 5)):
    """The order in which the ROIAlign kernels walk ``proposals`` [B,N,4] (level by level, top to bottom, so that ROIs
    reading the same feature pixels run close in time): int32 [B*N], a permutation of the row indices. Every
    ``pyramid_roi_align`` call computes it itself; a caller that pools the same proposals with several pool shapes computes
    it once and passes it as ``order=`` (N <= 4096 per image)."""
    levels = [int(v) for v in levels]
    rois = _lib.as_cuda(proposals, torch.float32)
    order = torch.empty((rois.shape[0] * rois.shape[1],), dtype=torch.int32, device=rois.device)
    dl = _lib.DL()
    _lib.check(_lib.lib().od_roi_processing_order(dl(rois), int(image_shape[0]), int(image_shape[1]), min(levels), len(levels),
                                                  dl(order), _lib.stream_ptr(rois.device)), "od_roi_processing_order")
    return order


def _map_dtype(maps):
    """The dtype the kernels read ``maps`` in: bfloat16 (no copy) when they are all bfloat16 CUDA tensors that the
    bf16 kernels take as they are (D % 8 == 0, 16-byte aligned data); float32 for anything else, converted as for host
    arrays (fp32 CUDA maps pass through unchanged), so that every map the fp32 path accepted is still accepted."""
    return _lib.read_dtype(maps, 16, depth_multiple=8)


def pyramid_roi_align(feature_maps, proposals, image_shape, pool_shape, levels=(2, 3, 4, 5), out=None,
                      return_levels=False, order=None, out_dtype=None):
    """FPN level assignment + bilinear crop_and_resize, one sample per bin (maskrcnn.py:104-187).

    feature_maps: list of [B,H_l,W_l,D] NHWC tensors for the ascending, contiguous ``levels``: float32 or bfloat16
    CUDA tensors are read as they are, anything else is converted to float32; proposals: [B,N,4] normalised
    (y1,x1,y2,x2). Returns pooled [1,B*N,ph,pw,D] (row b*N+n <-> proposals[b,n]) and, if requested, roi_level [B,N]
    int32. ``order``: optional result of ``roi_processing_order(proposals, ...)`` (saves the call's own pre-pass; the
    pooled values do not depend on it). The pooled dtype is ``out.dtype`` when ``out`` is given, else ``out_dtype``
    (float32 by default; bfloat16 is the round-to-nearest-even of the float32 result). bfloat16 maps or output need
    D % 8 == 0. The blend is float32 either way, so pooling bfloat16 maps equals pooling ``[f.float() for f in maps]``.
    """
    levels = [int(v) for v in levels]
    if levels != list(range(min(levels), min(levels) + len(levels))) or len(levels) != len(feature_maps):
        raise ValueError("levels must be ascending, contiguous and match feature_maps")
    rois = _lib.as_cuda(proposals, torch.float32)
    dev = rois.device
    map_dtype = _map_dtype(feature_maps)
    fmaps = [_lib.as_cuda(f, map_dtype, dev) for f in feature_maps]
    B, N = rois.shape[0], rois.shape[1]
    D = fmaps[0].shape[-1]
    ph, pw = int(pool_shape[0]), int(pool_shape[1])
    if out is None:
        out = torch.empty((1, B * N, ph, pw, D), dtype=out_dtype or torch.float32, device=dev)
    lv = torch.empty((B, N), dtype=torch.int32, device=dev) if return_levels else None
    dl = _lib.DL()
    ptrs = (ctypes.c_void_p * len(fmaps))(*[dl(f) for f in fmaps])
    L = _lib.lib()
    ws = _lib.zeroed_workspace(L.od_pyramid_roi_align_workspace_bytes_n(B * N), dev)   # ticket counter (stays zeroed) + ROI order
    od = _lib.as_cuda(order, torch.int32, dev) if order is not None else None
    _lib.check(L.od_pyramid_roi_align_forward_ordered(ptrs, len(fmaps), min(levels), dl(rois), int(image_shape[0]),
                                                      int(image_shape[1]), ph, pw, dl(out), dl(lv), dl(od), ws.data_ptr(),
                                                      ws.numel(), _lib.stream_ptr(dev)), "od_pyramid_roi_align_forward_ordered")
    return (out, lv) if return_levels else out


def crop_and_resize(image, boxes, box_ind, crop_size, extrapolation_value=0.0, out=None, out_dtype=None):
    """tf.image.crop_and_resize(method='bilinear') on an NHWC CUDA tensor: float32 or bfloat16 is read as it is,
    anything else is converted to float32. The output dtype is ``out.dtype`` when ``out`` is given, else ``out_dtype``
    (float32 by default); see ``pyramid_roi_align`` for the bfloat16 rules."""
    img = _lib.as_cuda(image, _map_dtype([image]))
    dev = img.device
    bx = _lib.as_cuda(boxes, torch.float32, dev)
    bi = _lib.as_cuda(box_ind, torch.int32, dev)
    ch, cw = int(crop_size[0]), int(crop_size[1])
    if out is None:
        out = torch.zeros((bx.shape[0], ch, cw, img.shape[-1]), dtype=out_dtype or torch.float32, device=dev)
    dl = _lib.DL()
    _lib.check(_lib.lib().od_crop_and_resize(dl(img), dl(bx), dl(bi), ch, cw, float(extrapolation_value), dl(out),
                                             _lib.stream_ptr(dev)), "od_crop_and_resize")
    return out


class MaskRCNN():
    # dtype of the pooled rows: None (float32) or torch.bfloat16. A class attribute, so that the constructor keeps the
    # reference signature: a bf16 head sets it on a subclass.
    pooled_dtype = None

    def __init__(self, image_shape, pool_shape, num_classes, levels, proposals, feature_maps, type='keras',
                 DEBUG=False):
        '''
        :param image_shape:   e.g. [1024, 1024, 3]
        :param pool_shape:    [7, 7] (or [14, 14] for the mask branch)
        :param num_classes:   kept for signature parity (only the dense head used it)
        :param levels:        [2, 3, 4, 5]
        :param proposals:     [num_batch, num_proposals, (y1, x1, y2, x2)] normalised
        :param feature_maps:  [P2, P3, P4, P5], each [num_batch, H, W, 256] NHWC, float32 or bfloat16
        '''
        self.image_shape = image_shape[0:2]
        self.pool_shape = pool_shape
        self.num_classes = num_classes
        self.levels = levels
        self.DEBUG = DEBUG
        self.build(proposals, feature_maps, type)

    def build(self, proposals, feature_maps, type='keras'):
        self.roi_pooling(self.image_shape, self.pool_shape, self.levels, proposals, feature_maps)

    def roi_pooling(self, image_shape, pool_shape, levels, proposals, feature_maps):
        """maskrcnn.py:74-187. The reference's per-level where/gather, concat and re-sort are fused away: each
        ROI is written straight to row b*N+n, and ``roi_level`` is the only one of the four DEBUG tensors that is
        data. ``box_to_level`` / ``sorting_tensor`` / ``ix`` (maskrcnn.py:128-173) are pure index plumbing - functions
        of ``roi_level`` - and are synthesised from it when DEBUG is set, with the reference's shapes and dtypes."""
        res = pyramid_roi_align(feature_maps, proposals, image_shape, pool_shape, levels, return_levels=self.DEBUG,
                                out_dtype=self.pooled_dtype)
        if self.DEBUG:
            self.pooled_rois, self.roi_level = res
            per_level = [torch.nonzero(self.roi_level == int(lv)) for lv in levels]         # tf.where: row-major
            b2l = torch.cat(per_level, dim=0).to(torch.int32)                               # [B*N, (batch, box)]
            box_range = torch.arange(b2l.shape[0], dtype=torch.int32, device=b2l.device)[:, None]
            self.box_to_level = torch.cat([b2l, box_range], dim=1)                          # maskrcnn.py:161-163
            self.sorting_tensor = self.box_to_level[:, 0] * 100000 + self.box_to_level[:, 1]   # maskrcnn.py:168
            # top_k(k = all).indices[::-1] (:171): descending with ties to the lower position, then reversed
            order = torch.sort(-self.sorting_tensor.to(torch.int64), stable=True).indices
            self.ix = torch.flip(order, dims=[0]).to(torch.int32)
        else:
            self.pooled_rois, self.roi_level = res, []
            self.box_to_level, self.sorting_tensor, self.ix = [], [], []

    def get_pooled_rois(self):
        return self.pooled_rois

    def get_mrcnn_graph(self):
        raise NotImplementedError("the dense classifier head (maskrcnn.py:189-315) is outside the detection-head "
                                  "hot path; feed its outputs (mrcnn_class_probs, mrcnn_bbox) to DetectionLayer")

    def debug_outputs(self):
        return self.roi_level, self.box_to_level, self.sorting_tensor, self.ix, None, None, None
