"""DetectionTargetLayer with the reference's interface
(MaskRCNN/building_blocks/data_processor.py:430-658, class BuildDetectionTargets)."""
from __future__ import annotations

import ctypes

import torch

from . import _lib
from .proposals import _stddev4


def _mask_dtype(gt_masks) -> torch.dtype:
    """The dtype od_detection_target_forward reads ``gt_masks`` in: bool or uint8 for a bool or uint8 tensor or numpy
    array, float32 for anything else."""
    import numpy as np
    if isinstance(gt_masks, torch.Tensor):
        dt = gt_masks.dtype
    elif isinstance(gt_masks, np.ndarray):
        dt = {np.dtype(np.bool_): torch.bool, np.dtype(np.uint8): torch.uint8}.get(gt_masks.dtype)
    else:
        dt = None
    return dt if dt in (torch.bool, torch.uint8) else torch.float32


class BuildDetectionTargets():
    """Proposal <-> GT IoU, positive/negative sampling, GT assignment, box-delta targets, zero padding.

    ``BuildDetectionTargets(conf, proposals, gt_class_ids, gt_bboxes, DEBUG=False)`` is per image like the
    reference (proposals [N,4], gt_class_ids [G], gt_bboxes [G,4]); a leading batch dimension on all three runs
    the whole batch in one launch (the batched generalisation of training.py:66-81).

    ``tf.random_shuffle`` (data_processor.py:587,:597) is unseeded in the reference. Here the two shuffles are
    driven by explicit permutations ``perm_pos`` / ``perm_neg`` ([N] or [B,N] int32 permutations of 0..N-1): the
    shuffled list is ``list[q]`` for q in perm (in order) with q < len(list). If omitted they are drawn with
    ``torch.randperm`` from ``generator`` (or the global CUDA RNG).
    """

    def __init__(self, conf, proposals, gt_class_ids, gt_bboxes, DEBUG=False, perm_pos=None, perm_neg=None,
                 generator=None, gt_masks=None):
        self.train_rois_per_image = conf.MRCNN_TRAIN_ROIS_PER_IMAGE
        self.box_stddev = conf.BBOX_STD_DEV
        self.mask_shape = tuple(getattr(conf, "MASK_SHAPE", (28, 28)))
        self.use_mini_mask = bool(getattr(conf, "USE_MINI_MASK", True))
        self.DEBUG = bool(DEBUG)
        self.roi_gt_masks = None
        self.build_detection_target(proposals, gt_class_ids, gt_bboxes, perm_pos, perm_neg, generator, gt_masks)

    def build_detection_target(self, proposals, gt_class_ids, gt_bboxes, perm_pos=None, perm_neg=None, generator=None,
                               gt_masks=None):
        L = _lib.lib()
        props = _lib.as_cuda(proposals, torch.float32)
        dev = props.device
        cls = _lib.as_cuda(gt_class_ids, torch.int32, dev)
        gtb = _lib.as_cuda(gt_bboxes, torch.float32, dev)
        single = props.dim() == 2
        if single:
            props, cls, gtb = props[None], cls[None], gtb[None]
        B, N = props.shape[0], props.shape[1]
        if N == 0:
            raise ValueError("roi_assertion: proposals must not be empty")   # tf.Assert, data_processor.py:550-555
        G, R = cls.shape[1], int(self.train_rois_per_image)

        def perm(p):
            if p is None:
                return torch.stack([torch.randperm(N, device=dev, generator=generator) for _ in range(B)]).to(torch.int32)
            p = _lib.as_cuda(p, torch.int32, dev)
            return p[None] if p.dim() == 1 else p
        pp, pn = perm(perm_pos).contiguous(), perm(perm_neg).contiguous()
        rois = torch.empty((B, R, 4), dtype=torch.float32, device=dev)
        rcls = torch.empty((B, R), dtype=torch.int32, device=dev)
        deltas = torch.empty((B, R, 4), dtype=torch.float32, device=dev)
        # optional mask targets: gt_masks in the reference's batch layout [B,Mh,Mw,G] ([Mh,Mw,G] per image,
        # data_processor.py:386,399); MINI_MASK_SHAPE masks cropped to their GT box when conf.USE_MINI_MASK.
        # bool and uint8 masks (what mask datasets store) stay one byte per element, on the host-to-device copy too:
        # the kernel widens each byte exactly, so the targets are those of gt_masks.float(). Other dtypes go as float32.
        masks = mtargets = None
        if gt_masks is not None:
            masks = _lib.as_cuda(gt_masks, _mask_dtype(gt_masks), dev)
            if single:
                masks = masks[None]
            if masks.dim() != 4 or masks.shape[0] != B or masks.shape[3] != G:
                raise ValueError("gt_masks must be [batch, mask_h, mask_w, max_gt_objects]")
            mtargets = torch.empty((B, R, int(self.mask_shape[0]), int(self.mask_shape[1])), dtype=torch.float32, device=dev)
        params = _lib.TargetParams(R, _stddev4(self.box_stddev), int(self.mask_shape[0]), int(self.mask_shape[1]),
                                   1 if self.use_mini_mask else 0, 1)
        dl = _lib.DL()
        dbg = _lib.TargetDebug()
        if self.DEBUG:
            d = dict(iou=torch.full((B, N, G), float("nan"), dtype=torch.float32, device=dev),
                     roi_iou_max=torch.full((B, N), float("nan"), dtype=torch.float32, device=dev),
                     pos_indices=torch.empty((B, N), dtype=torch.int32, device=dev),
                     neg_indices=torch.empty((B, N), dtype=torch.int32, device=dev),
                     counts=torch.empty((B, 6), dtype=torch.int32, device=dev),
                     sampled_pos=torch.empty((B, R), dtype=torch.int32, device=dev),
                     sampled_neg=torch.empty((B, R), dtype=torch.int32, device=dev),
                     gt_assignment=torch.empty((B, R), dtype=torch.int32, device=dev))
            for k, v in d.items():
                setattr(dbg, k, dl(v))
            self.debug_raw = d
        ws = _lib.workspace(L.od_detection_target_workspace_bytes(B, N, G), dev)
        _lib.check(L.od_detection_target_forward(dl(props), dl(cls), dl(gtb), dl(pp), dl(pn), ctypes.byref(params),
                                                 dl(rois), dl(rcls), dl(deltas), dl(masks), dl(mtargets), ctypes.byref(dbg),
                                                 ws.data_ptr(), ws.numel(), _lib.stream_ptr(dev)),
                   "od_detection_target_forward")
        if mtargets is not None:
            self.roi_gt_masks = mtargets[0] if single else mtargets
        if single:
            self.rois, self.roi_gt_class_ids, self.roi_gt_box_deltas = rois[0], rcls, deltas[0]   # cls is [1,R] (:627)
        else:
            self.rois, self.roi_gt_class_ids, self.roi_gt_box_deltas = rois, rcls, deltas
        if self.DEBUG:
            per_image = [self._reference_debug_dict(b, props[b], cls[b], gtb[b], rois[b], rcls[b], deltas[b])
                         for b in range(B)]
            self.debug_dict = per_image[0] if single else per_image

    def _reference_debug_dict(self, b, props, gt_cls, gt_box, rois, rcls, deltas):
        """The 21 named intermediates of data_processor.py:629-652 for image ``b``, with the reference's shapes and
        dtypes, assembled (DEBUG only; this synchronises) from what the kernel recorded: the IoU matrix in compacted
        row/column order, its row maxima, the sampled index lists, the GT assignment and the counts. As in the
        reference, ``pos_indices_05more`` / ``neg_indices_05more`` alias the lists AFTER shuffling + truncation (the
        variable is reassigned at :587 / :597 before the dict is built)."""
        raw = self.debug_raw
        n_prop, n_gt, _, _, pos_count, neg_count = (int(v) for v in raw["counts"][b].tolist())
        nzp = (props != 0).any(dim=1)                           # cast(reduce_sum(abs(p)), bool), :564
        nzg = gt_cls != 0                                       # :568
        sp = raw["sampled_pos"][b, :pos_count].to(torch.int64)
        sn = raw["sampled_neg"][b, :neg_count].to(torch.int64)
        iou = raw["iou"][b, :n_prop, :n_gt]
        assign = raw["gt_assignment"][b, :pos_count].to(torch.int64)
        gt_boxes_nz, gt_cls_nz = gt_box[nzg], gt_cls[nzg]
        R = int(self.train_rois_per_image)
        one_third = torch.tensor(1 / 0.33, dtype=torch.float32)          # float32(1/0.33) * float32(pos_count), :593
        neg_cnt = int((one_third * torch.tensor(float(pos_count), dtype=torch.float32)).to(torch.int32)) - pos_count
        return dict(
            non_zero_proposals=nzp, prop_corresponding_gt_non_zero=props[nzp], non_zeros_gt_box=nzg,
            gt_boxes_non_zero=gt_boxes_nz, gt_class_ids_non_zero=gt_cls_nz, iou=iou,
            roi_iou_max=raw["roi_iou_max"][b, :n_prop], pos_indices_05more=sp, neg_indices_05more=sn,
            num_pos_inst=int(R * 0.33), pos_indices=sp,
            pos_count=torch.tensor(pos_count, dtype=torch.int32), neg_cnt=torch.tensor(neg_cnt, dtype=torch.int32),
            neg_indices=sn, pos_rois=rois[:pos_count], neg_rois=rois[pos_count:pos_count + neg_count],
            pos_iou=iou[sp], roi_gt_box_assignment=assign, roi_gt_class_ids=rcls[:pos_count],
            roi_gt_boxes=gt_boxes_nz[assign], roi_gt_box_deltas=deltas[:pos_count])

    def get_target_rois(self):
        return self.rois, self.roi_gt_class_ids, self.roi_gt_box_deltas

    def get_target_masks(self):
        """[R,mask_h,mask_w] ([B,R,...] batched) mask targets of the sampled positives (zero rows elsewhere); only
        built when ``gt_masks`` was given. North-star extension - the reference never builds them."""
        return self.roi_gt_masks

    def debug_outputs(self):
        """The reference's debug dict (data_processor.py:629-652, 21 keys) - one dict for a per-image call, a list of
        dicts for a batched one. ``debug_raw`` keeps the kernel's own batched arrays (pre-shuffle index lists,
        counts [B,6], ...)."""
        return self.debug_dict


class PreprareTrainData():
    """RPN-target part of the reference's training data preparer (data_processor.py:110-294; the class name keeps
    the reference's spelling). ``PreprareTrainData(conf, dataset=None)`` builds the pixel-coordinate anchors once
    (:129-140, on the GPU, bit-exact with numpy) and ``build_rpn_targets(batch_gt_boxes)`` labels them against one
    image's GT boxes exactly like the reference's float64 numpy code (:173-294) - on the device, in float64.

    The image molding / mask resizing / batch assembly methods of the reference class are host data-pipeline code
    outside the detection-head path and are not part of this package.

    ``np.random.choice(idx, extra, replace=False)`` (:246, :253) is unseeded in the reference. Here the two draws are
    explicit permutations ``perm_pos`` / ``perm_neg`` of ``0..A-1``: with ``idx = where(label == +1 / -1)``, the entries
    ``idx[q]`` for the first ``extra`` values ``q`` of the permutation with ``q < len(idx)`` are reset to 0. (numpy's
    legacy ``choice`` takes ``permutation(len(idx))[:extra]``, so a permutation that starts with that draw reproduces
    the reference bit for bit - see tests/golden/make_golden_rpn.py.) Omitted permutations come from ``torch.randperm``.
    """

    def __init__(self, conf, dataset=None, device=None):
        from . import utils
        self.conf = conf
        self.dataset = dataset
        self.max_rpn_targets = conf.RPN_TRAIN_ANCHORS_PER_IMAGE
        self.bbox_std_dev = conf.RPN_BBOX_STDDEV
        feature_shapes = utils.get_resnet_stage_shapes(conf, conf.IMAGE_SHAPE)
        self.anchors = utils.gen_anchors_pixel_coord(conf.RPN_ANCHOR_SCALES, conf.RPN_ANCHOR_RATIOS, feature_shapes,
                                                     conf.RESNET_STRIDES, conf.RPN_ANCHOR_STRIDE, device=device)
        self.anchor_area = (self.anchors[:, 2] - self.anchors[:, 0]) * (self.anchors[:, 3] - self.anchors[:, 1])

    def build_rpn_targets(self, batch_gt_boxes, perm_pos=None, perm_neg=None, generator=None, gt_count=None,
                          return_counts=False):
        """batch_gt_boxes: [num_objects, (y1,x1,y2,x2)] pixels for ONE image (the reference's form) -> returns
        (positive_anchors [num_pos,4] f64, rpn_target_class [A] i32, rpn_target_bbox [max_rpn_targets,4] f64).
        A 3-D [B,G,4] input (with ``gt_count`` [B], default G) runs the batch in one call and returns the padded
        tensors ([B,max,4], [B,A], [B,max,4]) plus counts [B,4] when ``return_counts``."""
        L = _lib.lib()
        anchors = self.anchors
        dev = anchors.device
        gt = _lib.as_cuda(batch_gt_boxes, torch.float64, dev)
        single = gt.dim() == 2
        if single:
            gt = gt[None]
        B, G = gt.shape[0], gt.shape[1]
        A, T = anchors.shape[0], int(self.max_rpn_targets)
        if gt_count is None:
            cnt = torch.full((B,), G, dtype=torch.int32, device=dev)
        else:
            cnt = _lib.as_cuda(gt_count, torch.int32, dev).reshape(B)

        def perm(p):
            if p is None:
                return torch.stack([torch.randperm(A, device=dev, generator=generator) for _ in range(B)]).to(torch.int32)
            p = _lib.as_cuda(p, torch.int32, dev)
            return (p[None] if p.dim() == 1 else p).contiguous()
        pp, pn = perm(perm_pos), perm(perm_neg)
        cls = torch.empty((B, A), dtype=torch.int32, device=dev)
        bbox = torch.empty((B, T, 4), dtype=torch.float64, device=dev)
        pos = torch.empty((B, T, 4), dtype=torch.float64, device=dev)
        counts = torch.empty((B, 4), dtype=torch.int32, device=dev)
        sd = [float(v) for v in self.bbox_std_dev]
        params = _lib.RpnTargetParams(T, (ctypes.c_double * 4)(*sd))
        ws = _lib.workspace(L.od_rpn_target_workspace_bytes(B, A, G), dev)
        dl = _lib.DL()
        _lib.check(L.od_rpn_target_forward(dl(anchors), dl(gt.contiguous()), dl(cnt), dl(pp), dl(pn), ctypes.byref(params),
                                           dl(cls), dl(bbox), dl(pos), dl(counts), ws.data_ptr(), ws.numel(),
                                           _lib.stream_ptr(dev)), "od_rpn_target_forward")
        if single:
            n_pos = int(counts[0, 2].item())          # like the reference: positive_anchors has one row per positive
            out = (pos[0, :n_pos], cls[0], bbox[0])
        else:
            out = (pos, cls, bbox)
        return out + (counts,) if return_counts else out
