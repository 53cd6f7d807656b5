"""CPU ORACLE — test infrastructure only.

ctypes front-end of ``oracle/odhead_oracle.c`` (the C restatement of the
reference's detection-head algorithm) working on numpy arrays.  Only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl
reference`` legs may import this package; ``objectdetection_b200`` never does.

Parity status: see the header of ``odhead_oracle.c`` — the numpy-only helpers are
pinned by the reference's own functions (``tests/golden``); the three TensorFlow
kernels are anchored to TensorFlow's published kernel-test vectors
(``tests/test_tf_known_answers.py``); the four layers composed from them are
**parity unpinned** (TensorFlow is not installable here and the reference records
no outputs for those layers).
"""
from __future__ import annotations

import ctypes
import hashlib
import os
import subprocess
import tempfile
from ctypes import POINTER, c_double, c_float, c_int32, c_int64, c_void_p

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "odhead_oracle.c")
_LIB = os.path.join(_HERE, "liboracle.so")
_lib = None


def _built_from(lib: str, digest: str) -> bool:
    try:
        with open(lib + ".sha1") as f:
            return f.read().strip() == digest and os.path.exists(lib)
    except OSError:
        return False


def _private_dir(digest: str) -> str:
    """One directory per user and source under the system's temporary directory, shared by every process that
    needs the library while the tree is read-only."""
    d = os.path.join(tempfile.gettempdir(), f"oracle-{os.getuid()}-{digest[:16]}")
    os.makedirs(d, mode=0o700, exist_ok=True)
    st = os.stat(d)
    if st.st_uid != os.getuid() or st.st_mode & 0o022:
        raise RuntimeError(f"{d} exists and is not a private directory of this user")
    return d


def build(force: bool = False) -> str:
    """Compile ``liboracle.so`` next to its source (gcc, no FMA contraction).

    A library is up to date when its stamp (``liboracle.so.sha1``) holds the sha1 of the source it was built from;
    file times are not used, a copy of the tree does not keep them. In a read-only tree a missing or stale library is
    built once per source in a directory under the system's temporary directory, which ``_LIB`` then names."""
    global _LIB
    if not os.path.exists(_SRC):
        return _LIB
    with open(_SRC, "rb") as f:
        digest = hashlib.sha1(f.read()).hexdigest()
    out = os.path.join(_HERE, "liboracle.so")
    if not force and _built_from(out, digest):
        _LIB = out
        return out
    if not os.access(_HERE, os.W_OK):
        out = os.path.join(_private_dir(digest), "liboracle.so")
        if not force and _built_from(out, digest):
            _LIB = out
            return out
    part = f"{out}.{os.getpid()}.part"       # renamed into place: a concurrent process never loads half a library
    base = ["-O2", "-std=c11", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math",
            "-fvisibility=hidden", "-o", part, _SRC, "-lm"]
    errors = []
    for cc in ("/usr/bin/gcc", "gcc", "cc"):
        for omp in (["-fopenmp"], []):
            try:
                subprocess.run([cc] + omp + base, check=True, capture_output=True, text=True)
            except (subprocess.CalledProcessError, FileNotFoundError) as e:  # try next
                errors.append(f"{cc} {' '.join(omp)}: {getattr(e, 'stderr', e)}")
                continue
            os.replace(part, out)
            with open(out + ".sha1", "w") as f:
                f.write(digest)
            _LIB = out
            return out
    raise RuntimeError("could not build the oracle:\n" + "\n".join(errors))


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        build()
        _lib = ctypes.CDLL(_LIB)
        _lib.orc_tf_iou.restype = c_float
        _lib.orc_target_iou.restype = c_float
        _lib.orc_nms.restype = c_int32
        _lib.orc_roi_level.restype = c_int32
        _lib.orc_detection_targets.restype = c_int32
        _lib.orc_anchor_count.restype = c_int64
        _lib.orc_frcnn_nms_sorted.restype = c_int32
        _lib.orc_frcnn_proposals.restype = c_int32
    return _lib


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def _p(a):
    return None if a is None else a.ctypes.data_as(c_void_p)


# --------------------------------------------------------------------------- ops
def topk(scores: np.ndarray, k: int):
    """tf.nn.top_k(sorted=True) over the last axis of a 2-D float32 array (any strides)."""
    assert scores.ndim == 2 and scores.dtype == np.float32
    rows, cols = scores.shape
    rs, cs = (s // 4 for s in scores.strides)
    idx = np.empty((rows, k), np.int32)
    val = np.empty((rows, k), np.float32)
    lib().orc_topk(_p(scores), c_int64(rows), c_int64(cols), c_int64(rs), c_int64(cs), c_int64(k),
                   _p(idx), _p(val))
    return val, idx


def apply_box_deltas(boxes, deltas):
    boxes, deltas = _f32(boxes), _f32(deltas)
    out = np.empty_like(boxes)
    lib().orc_apply_box_deltas(_p(boxes), _p(deltas), c_int64(boxes.size // 4), _p(out))
    return out


def clip_boxes(boxes, window):
    """window: [4] shared or [B,4] per leading-batch entry of boxes [B,K,4]."""
    boxes, window = _f32(boxes), _f32(window)
    out = np.empty_like(boxes)
    if window.ndim == 1:
        lib().orc_clip_boxes(_p(boxes), _p(window), c_int64(boxes.size // 4), _p(out))
    else:
        for b in range(boxes.shape[0]):
            bb = np.ascontiguousarray(boxes[b])
            ob = np.empty_like(bb)
            lib().orc_clip_boxes(_p(bb), _p(np.ascontiguousarray(window[b])), c_int64(bb.size // 4), _p(ob))
            out[b] = ob
    return out


def tf_iou(bi, bj) -> float:
    bi, bj = _f32(bi), _f32(bj)
    return float(lib().orc_tf_iou(_p(bi), _p(bj)))


def target_iou(p, g) -> float:
    p, g = _f32(p), _f32(g)
    return float(lib().orc_target_iou(_p(p), _p(g)))


def nms(boxes, scores, max_out: int, thr: float) -> np.ndarray:
    """tf.image.non_max_suppression: returns kept indices in selection order."""
    boxes, scores = _f32(boxes).reshape(-1, 4), _f32(scores).reshape(-1)
    n = boxes.shape[0]
    keep = np.empty(max(max_out, 1), np.int32)
    cnt = lib().orc_nms(_p(boxes), _p(scores), c_int32(n), c_int32(max_out), c_float(thr), _p(keep))
    return keep[:cnt].copy()


def crop_and_resize(image, boxes, box_ind, crop_h: int, crop_w: int, extrapolation: float = 0.0, out=None):
    image, boxes, box_ind = _f32(image), _f32(boxes).reshape(-1, 4), _i32(box_ind).reshape(-1)
    B, H, W, D = image.shape
    n = boxes.shape[0]
    if out is None:
        out = np.zeros((n, crop_h, crop_w, D), np.float32)
    lib().orc_crop_and_resize(_p(image), c_int32(B), c_int32(H), c_int32(W), c_int32(D), _p(boxes), _p(box_ind),
                              c_int32(n), c_int32(crop_h), c_int32(crop_w), c_float(extrapolation), _p(out))
    return out


def roi_level(rois, image_h: int, image_w: int, min_level: int = 2, max_level: int = 5) -> np.ndarray:
    rois = _f32(rois)
    flat = rois.reshape(-1, 4)
    out = np.empty(flat.shape[0], np.int32)
    L = lib()
    for i in range(flat.shape[0]):
        out[i] = L.orc_roi_level(_p(flat[i]), c_int32(image_h), c_int32(image_w), c_int32(min_level), c_int32(max_level))
    return out.reshape(rois.shape[:-1])


def pyramid_roi_align(fmaps, rois, image_h: int, image_w: int, pool_h: int, pool_w: int, min_level: int = 2):
    """MaskRCNN.roi_pooling: returns (pooled [1,B*N,ph,pw,D], roi_level [B,N])."""
    fmaps = [_f32(f) for f in fmaps]
    rois = _f32(rois)
    B, N = rois.shape[:2]
    D = fmaps[0].shape[-1]
    L = len(fmaps)
    ptrs = (c_void_p * L)(*[f.ctypes.data for f in fmaps])
    fh = _i32([f.shape[1] for f in fmaps])
    fw = _i32([f.shape[2] for f in fmaps])
    out = np.zeros((B * N, pool_h, pool_w, D), np.float32)
    lv = np.empty((B, N), np.int32)
    lib().orc_pyramid_roi_align(ptrs, _p(fh), _p(fw), c_int32(L), c_int32(min_level), c_int32(B), c_int32(D),
                                _p(rois), c_int32(N), c_int32(image_h), c_int32(image_w),
                                c_int32(pool_h), c_int32(pool_w), _p(out), _p(lv))
    return out[None], lv


def proposal_forward(probs, bbox, anchors, stddev, pre_nms_limit: int, post_nms_count: int, nms_thr: float,
                     debug: bool = False):
    """Proposals.build. Returns proposals [B,N,4] (and a dict of intermediates if debug)."""
    probs, bbox, anchors = _f32(probs), _f32(bbox), _f32(anchors)
    B, A = probs.shape[:2]
    K, N = min(pre_nms_limit, A), post_nms_count
    stddev = _f32(stddev)
    out = np.empty((B, N, 4), np.float32)
    d = None
    if debug:
        d = dict(ix=np.empty((B, K), np.int32), scores=np.empty((B, K), np.float32),
                 bbox_delta=np.empty((B, K, 4), np.float32), anchors=np.empty((B, K, 4), np.float32),
                 anchor_delta=np.empty((B, K, 4), np.float32), anchor_delta_clipped=np.empty((B, K, 4), np.float32),
                 keep_idx=np.empty((B, N), np.int32), num_kept=np.empty((B,), np.int32))
    g = (lambda k: _p(d[k])) if debug else (lambda k: None)
    lib().orc_proposal_forward(_p(probs), _p(bbox), _p(anchors), c_int32(B), c_int32(A), _p(stddev),
                               c_int32(pre_nms_limit), c_int32(N), c_float(nms_thr), _p(out),
                               g("ix"), g("scores"), g("bbox_delta"), g("anchors"), g("anchor_delta"),
                               g("anchor_delta_clipped"), g("keep_idx"), g("num_kept"))
    return (out, d) if debug else out


def rpn_levels_to_flat(class_logits_levels, bbox_levels):
    """The RPN head's output plumbing (numpy): each level's conv outputs [B,H,W,2a] / [B,H,W,4a] are reshaped to
    [B,-1,2] / [B,-1,4] (rpn.py:54-55, :66), the (bg, fg) pairs go through a softmax (rpn.py:58-59; tf.nn.softmax =
    exp(x - max) / sum, fp32, exp rounded from fp64 like everywhere in this oracle) and the levels are concatenated
    along the anchor axis (training.py:163-166). Returns (rpn_class_probs [B,A,2], rpn_bbox [B,A,4])."""
    probs, boxes = [], []
    for c, d in zip(class_logits_levels, bbox_levels):
        c, d = _f32(c), _f32(d)
        x = c.reshape(c.shape[0], -1, 2)
        m = x.max(axis=-1, keepdims=True)
        e = np.exp((x - m).astype(np.float64)).astype(np.float32)
        probs.append(e / (e[..., :1] + e[..., 1:]))
        boxes.append(d.reshape(d.shape[0], -1, 4))
    return np.concatenate(probs, axis=1), np.concatenate(boxes, axis=1)


def detection_targets(proposals, gt_class_ids, gt_boxes, perm_pos, perm_neg, rois_per_image: int, stddev):
    """BuildDetectionTargets for ONE image. Returns (rois [R,4], cls [1,R], deltas [R,4], debug dict)."""
    proposals, gt_boxes = _f32(proposals), _f32(gt_boxes)
    gt_class_ids, perm_pos, perm_neg = _i32(gt_class_ids), _i32(perm_pos), _i32(perm_neg)
    N, G, R = proposals.shape[0], gt_boxes.shape[0], rois_per_image
    stddev = _f32(stddev)
    rois = np.empty((R, 4), np.float32)
    cls = np.empty((R,), np.int32)
    deltas = np.empty((R, 4), np.float32)
    dbg = dict(iou=np.full((N, G), np.nan, np.float32), roi_iou_max=np.full((N,), np.nan, np.float32),
               pos_indices=np.empty((N,), np.int32), neg_indices=np.empty((N,), np.int32),
               counts=np.empty((6,), np.int32), sampled_pos=np.empty((R,), np.int32),
               sampled_neg=np.empty((R,), np.int32), gt_assignment=np.empty((R,), np.int32))
    rc = lib().orc_detection_targets(_p(proposals), _p(gt_class_ids), _p(gt_boxes), c_int32(N), c_int32(G),
                                     _p(perm_pos), _p(perm_neg), c_int32(R), _p(stddev),
                                     _p(rois), _p(cls), _p(deltas), _p(dbg["iou"]), _p(dbg["roi_iou_max"]),
                                     _p(dbg["pos_indices"]), _p(dbg["neg_indices"]), _p(dbg["counts"]),
                                     _p(dbg["sampled_pos"]), _p(dbg["sampled_neg"]), _p(dbg["gt_assignment"]))
    if rc != 0:
        raise ValueError("pos_count + neg_count exceeds rois_per_image")
    return rois, cls[None], deltas, dbg


def mask_targets(rois, gt_class_ids, gt_boxes, gt_masks_hwg, dbg, mask_shape=(28, 28), use_mini_mask=True):
    """Mask targets of ONE image's sampled positives (north-star extension; **parity unpinned**: absent from the
    reference, whose mask head is commented out - masking.py:1-67 - restated from the model it re-writes, matterport
    Mask_RCNN ``detection_targets_graph``): ``round(crop_and_resize(gt_mask[assigned], box, mask_shape))`` with
    ``box`` = the ROI, re-expressed in the GT box's frame for mini masks. ``rois`` [R,4] and ``dbg`` come from
    ``detection_targets``; ``gt_masks_hwg`` is [Mh,Mw,G] (batch_gt_masks layout, data_processor.py:386).
    Returns [R,mh,mw] float32 (zero rows for non-positives)."""
    rois, gt_boxes = _f32(rois), _f32(gt_boxes)
    masks = _f32(gt_masks_hwg)
    R = rois.shape[0]
    mh, mw = int(mask_shape[0]), int(mask_shape[1])
    out = np.zeros((R, mh, mw), np.float32)
    pos_count = int(dbg["counts"][4])
    if pos_count == 0:
        return out
    valid = np.nonzero(_i32(gt_class_ids) != 0)[0]
    src = valid[dbg["gt_assignment"][:pos_count]]
    boxes = rois[:pos_count].copy()
    if use_mini_mask:
        gt = gt_boxes[src]
        gt_h = gt[:, 2] - gt[:, 0]
        gt_w = gt[:, 3] - gt[:, 1]
        with np.errstate(all="ignore"):
            boxes = np.stack([(boxes[:, 0] - gt[:, 0]) / gt_h, (boxes[:, 1] - gt[:, 1]) / gt_w,
                              (boxes[:, 2] - gt[:, 0]) / gt_h, (boxes[:, 3] - gt[:, 1]) / gt_w], axis=1).astype(np.float32)
    roi_masks = np.ascontiguousarray(np.transpose(masks, (2, 0, 1))[src][..., None])     # [n,Mh,Mw,1]
    crops = crop_and_resize(roi_masks, boxes, np.arange(pos_count, dtype=np.int32), mh, mw)
    out[:pos_count] = np.round(crops[..., 0])     # tf.round: half to even
    return out


def rpn_targets(anchors, gt_boxes, perm_pos, perm_neg, max_rpn_targets: int, stddev):
    """PreprareTrainData.build_rpn_targets (data_processor.py:173-294) for ONE image, numpy float64 like the reference,
    with utils.intersection_over_union (utils.py:32-40). The two ``np.random.choice(idx, extra, replace=False)``
    draws (:246, :253) are explicit permutations: ``idx[q]`` is reset to 0 for the first ``extra`` entries ``q`` of the
    permutation with ``q < len(idx)``. Pinned by tests/golden/reference_rpn_targets.npz (the reference's own output).
    Returns (positive_anchors [n_pos,4], rpn_target_class [A] int32, rpn_target_bbox [max,4], counts [4])."""
    anchors = _f64(anchors)
    gt = _f64(gt_boxes)
    A = anchors.shape[0]
    cls = np.zeros([A], dtype="int32")
    anchor_area = (anchors[:, 2] - anchors[:, 0]) * (anchors[:, 3] - anchors[:, 1])
    gt_area = (gt[:, 2] - gt[:, 0]) * (gt[:, 3] - gt[:, 1])
    overlaps = np.zeros((gt.shape[0], A))
    for i in range(gt.shape[0]):
        y1 = np.maximum(gt[i, 0], anchors[:, 0])
        y2 = np.minimum(gt[i, 2], anchors[:, 2])
        x1 = np.maximum(gt[i, 1], anchors[:, 1])
        x2 = np.minimum(gt[i, 3], anchors[:, 3])
        inter = np.maximum(x2 - x1, 0) * np.maximum(y2 - y1, 0)
        overlaps[i] = inter / (gt_area[i] + anchor_area - inter)
    overlaps = overlaps.T
    if gt.shape[0] > 0:
        amax_idx = np.argmax(overlaps, axis=1)
        amax = overlaps[np.arange(A), amax_idx]
    else:                                   # (the reference cannot run without GT; all background here)
        amax_idx, amax = np.zeros(A, np.int64), np.zeros(A)
    cls[amax < 0.3] = -1
    if gt.shape[0] > 0:
        cls[np.argmax(overlaps, axis=0)] = 1
    cls[amax >= 0.7] = 1

    def drop(label, perm, extra):
        idx = np.where(cls == label)[0]
        if extra > 0:
            q = np.asarray(perm)[np.asarray(perm) < len(idx)][:extra]
            cls[idx[q]] = 0
    idx = np.where(cls == 1)[0]
    n_pos0 = len(idx)
    drop(1, perm_pos, n_pos0 - max_rpn_targets // 2)
    n_neg0 = int(np.sum(cls == -1))
    drop(-1, perm_neg, n_neg0 - (max_rpn_targets - int(np.sum(cls == 1))))
    bbox = np.zeros((max_rpn_targets, 4))
    pos_idx = np.where(cls == 1)[0]
    sd = _f64(stddev)
    for i, a in enumerate(pos_idx):
        g = gt[amax_idx[a]]
        an = anchors[a]
        ah, aw = an[2] - an[0], an[3] - an[1]
        acy, acx = an[0] + 0.5 * ah, an[1] + 0.5 * aw
        gh, gw = g[2] - g[0], g[3] - g[1]
        gcy, gcx = g[0] + 0.5 * gh, g[1] + 0.5 * gw
        bbox[i] = [(gcy - acy) / ah, (gcx - acx) / aw, np.log(gh / ah), np.log(gw / aw)]
        bbox[i] /= sd
    counts = np.array([n_pos0, n_neg0, len(pos_idx), int(np.sum(cls == -1))], np.int32)
    return anchors[pos_idx], cls, bbox, counts


def _exp32(x):
    return np.exp(np.asarray(x, np.float32).astype(np.float64)).astype(np.float32)


def _log32(x):
    return np.log(np.asarray(x, np.float32).astype(np.float64)).astype(np.float32)


def rpn_losses(rpn_target_class, rpn_class_logits, rpn_target_bbox, rpn_pred_box):
    """Loss.rpn_class_loss (loss_optimize.py:11-44) and Loss.rpn_box_loss (:47-87), numpy: per-element values in fp32
    in the reference's operation order, means over fp64 sums. Returns (class_loss, box_loss, rpn_pred_box_pos)."""
    tc = np.asarray(rpn_target_class).reshape(np.asarray(rpn_class_logits).shape[:2]).astype(np.int32)   # squeeze (:24)
    lg = _f32(rpn_class_logits)
    sel = tc != 0                                                   # tf.where(not_equal(., 0)) (:28)
    x = lg[sel]
    label = (tc[sel] == 1).astype(np.int64)                         # (:32)
    if x.shape[0]:
        m = x.max(-1)
        s = _exp32(x[:, 0] - m) + _exp32(x[:, 1] - m)
        ce = _log32(s) - (x[np.arange(x.shape[0]), label] - m)      # sparse_categorical_crossentropy(from_logits)
        class_loss = np.float32(ce.astype(np.float64).sum() / ce.shape[0])
    else:
        class_loss = np.float32(0.0)                                # K.switch (:42)
    tb, pb = _f32(rpn_target_bbox), _f32(rpn_pred_box)
    pos = tc == 1
    pred_pos = pb[pos]                                              # gather_nd over tf.where: (image, anchor) order (:63-64)
    T = tb.shape[1]
    tgt, prd = [], []
    for b in range(tb.shape[0]):
        n = int(pos[b].sum())                                       # non_pad_count (:68)
        tgt.append(tb[b, :min(n, T)])                               # rpn_target_bbox[i, :count] (:70-72)
        prd.append(pb[b][pos[b]][:min(n, T)])
    tgt, prd = np.concatenate(tgt, 0), np.concatenate(prd, 0)
    if tgt.size:
        d = np.abs(tgt - prd)
        less = (d < np.float32(1.0)).astype(np.float32)
        l = (np.float32(0.5) * less) * (d * d) + (d - np.float32(0.5)) * (np.float32(1.0) - less)   # (:79-81)
        box_loss = np.float32(l.astype(np.float64).sum() / l.size)
    else:
        box_loss = np.float32(0.0)
    return class_loss, box_loss, pred_pos


def mrcnn_losses(mrcnn_target_class_ids, mrcnn_pred_logits, batch_active_class_ids, mrcnn_target_box, mrcnn_pred_box):
    """Loss.mrcnn_class_loss (loss_optimize.py:89-151) and Loss.mrcnn_box_loss (:154-201), numpy.
    Returns (pred_active [B,R], class_loss, box_loss)."""
    ids = np.asarray(mrcnn_target_class_ids).astype(np.int64)
    lg, act = _f32(mrcnn_pred_logits), _f32(batch_active_class_ids)
    B, R, C = lg.shape
    # tf.argmax (:113) as a serial scan with a strict '>' (the rule of DetectionLayer's argmax too): the first maximum
    # wins and a NaN never replaces the running maximum, where np.argmax would return the first NaN
    pred_cls = np.zeros((B, R), np.int64)
    m = lg[..., 0].copy()
    for j in range(1, C):
        up = lg[..., j] > m
        pred_cls[up] = j
        m[up] = lg[..., j][up]
    pred_active = act[0][pred_cls]                                  # tf.gather(batch_active_class_ids[0], .) (:115)
    s = np.zeros((B, R), np.float32)
    for j in range(C):                                              # fp32 sum in class order
        s = s + _exp32(lg[..., j] - m)
    ce = _log32(s) - (np.take_along_axis(lg, ids[..., None], -1)[..., 0] - m)   # sparse_softmax_cross_entropy (:139-142)
    with np.errstate(invalid="ignore", divide="ignore"):
        class_loss = np.float32((ce * pred_active).astype(np.float64).sum() / pred_active.astype(np.float64).sum())
    tb, pb = _f32(mrcnn_target_box), _f32(mrcnn_pred_box)
    posm = ids > 0                                                  # (:171)
    t = tb[posm]
    p = pb[posm, ids[posm]]                                         # predicted box of the target class (:180-184)
    if t.size:
        eps = np.float32(1e-7)
        o = np.minimum(np.maximum(p, eps), np.float32(1.0) - eps)   # K.binary_crossentropy: clip, logit, sigmoid CE
        z = _log32(o / (np.float32(1.0) - o))
        l1p = np.log1p(_exp32(-np.abs(z)).astype(np.float64)).astype(np.float32)
        l = (np.maximum(z, np.float32(0.0)) - z * t) + l1p
        box_loss = np.float32(l.astype(np.float64).sum() / l.size)
    else:
        box_loss = np.float32(0.0)
    return pred_active, class_loss, box_loss


def detection_forward(proposals, probs, bbox, window_norm, stddev, min_conf: float, nms_thr: float,
                      max_instances: int, debug: bool = False):
    """DetectionLayer.build. Returns detections [B,M,6] (and intermediates if debug)."""
    proposals, probs, bbox, window_norm = _f32(proposals), _f32(probs), _f32(bbox), _f32(window_norm)
    B, N, C = probs.shape
    stddev = _f32(stddev)
    det = np.empty((B, max_instances, 6), np.float32)
    d = None
    if debug:
        d = dict(class_ids=np.empty((B, N), np.int32), class_scores=np.empty((B, N), np.float32),
                 refined_proposals=np.empty((B, N, 4), np.float32), clipped_proposals=np.empty((B, N, 4), np.float32),
                 keep_mask=np.empty((B, N), np.int32), nms_keep_mask=np.empty((B, N), np.int32))
    g = (lambda k: _p(d[k])) if debug else (lambda k: None)
    lib().orc_detection_forward(_p(proposals), _p(probs), _p(bbox), _p(window_norm), c_int32(B), c_int32(N),
                                c_int32(C), _p(stddev), c_float(min_conf), c_float(nms_thr), c_int32(max_instances),
                                _p(det), g("class_ids"), g("class_scores"), g("refined_proposals"),
                                g("clipped_proposals"), g("keep_mask"), g("nms_keep_mask"))
    return (det, d) if debug else det


# ----------------------------------------------------------------------- anchors
class AnchorSpec(ctypes.Structure):
    _fields_ = [("num_levels", c_int32), ("num_ratios", c_int32), ("scales", c_double * 8), ("ratios", c_double * 8),
                ("fmap_h", c_int32 * 8), ("fmap_w", c_int32 * 8), ("fmap_stride", c_int32 * 8),
                ("anchor_stride", c_int32), ("image_h", c_int32), ("image_w", c_int32)]


def anchor_spec(image_shape, scales, ratios, feature_map_shapes, feature_map_strides, anchor_stride) -> AnchorSpec:
    s = AnchorSpec()
    s.num_levels, s.num_ratios = len(scales), len(ratios)
    for i, v in enumerate(scales):
        s.scales[i] = float(v)
        s.fmap_h[i], s.fmap_w[i] = int(feature_map_shapes[i][0]), int(feature_map_shapes[i][1])
        s.fmap_stride[i] = int(feature_map_strides[i])
    for i, v in enumerate(ratios):
        s.ratios[i] = float(v)
    s.anchor_stride, s.image_h, s.image_w = int(anchor_stride), int(image_shape[0]), int(image_shape[1])
    return s


def gen_anchors(image_shape, batch_size, scales, ratios, feature_map_shapes, feature_map_strides, anchor_strides):
    """utils.gen_anchors: [B,A,4] float32 normalised."""
    s = anchor_spec(image_shape, scales, ratios, feature_map_shapes, feature_map_strides, anchor_strides)
    A = lib().orc_anchor_count(ctypes.byref(s))
    norm = np.empty((A, 4), np.float32)
    lib().orc_gen_anchors(ctypes.byref(s), None, _p(norm))
    return np.ascontiguousarray(np.broadcast_to(norm, (batch_size, A, 4)))


def gen_anchors_pixel_coord(scales, ratios, feature_map_shapes, feature_map_strides, anchor_strides):
    """utils.gen_anchors_pixel_coord: [A,4] float64 pixels."""
    s = anchor_spec((2, 2), scales, ratios, feature_map_shapes, feature_map_strides, anchor_strides)
    A = lib().orc_anchor_count(ctypes.byref(s))
    pix = np.empty((A, 4), np.float64)
    lib().orc_gen_anchors(ctypes.byref(s), _p(pix), None)
    return pix


def norm_boxes(box, img_shape):
    """utils.norm_boxes (utils.py:181-196): fp64 divide, cast to float32."""
    h, w = img_shape
    scale = np.array([h - 1, w - 1, h - 1, w - 1])
    shift = np.array([0, 0, 1, 1])
    return np.divide((np.asarray(box) - shift), scale).astype(np.float32)


def norm_boxes_tf(boxes, img_shape):
    """utils.norm_boxes_tf (utils.py:198-210), the in-graph fp32 normalisation of the GT boxes (training.py:135):
    scale = float32([h, w, h, w]) - 1.0f; (boxes - [0,0,1,1]) / scale, every operation in float32."""
    h, w = (np.float32(v) for v in img_shape)
    scale = np.array([h, w, h, w], np.float32) - np.float32(1.0)
    shift = np.array([0., 0., 1., 1.], np.float32)
    return (np.asarray(boxes, np.float32) - shift) / scale


def denorm_boxes(boxes, shape):
    """utils.denorm_boxes (utils.py:212-227)."""
    h, w = shape
    scale = np.array([h - 1, w - 1, h - 1, w - 1])
    shift = np.array([0, 0, 1, 1])
    return np.around(np.multiply(boxes, scale) + shift).astype(np.int32)


def get_resnet_stage_shapes(strides, image_shape):
    """utils.get_resnet_stage_shapes (utils.py:155-178)."""
    return np.array([[int(np.ceil(image_shape[0] / s)), int(np.ceil(image_shape[1] / s))] for s in strides])


def unmold_detection(original_image_shape, image_shape, detections, image_window):
    """detection.unmold_detection (detection.py:8-53), numpy like the reference."""
    image_window = norm_boxes(image_window, image_shape[:2])
    zero_ix = np.where(detections[:, 4] == 0)[0]
    n = zero_ix[0] if zero_ix.shape[0] > 0 else detections.shape[0]
    boxes = detections[:n, :4]
    class_ids = detections[:n, 4].astype(np.int32)
    scores = detections[:n, 5]
    wy1, wx1, wy2, wx2 = image_window
    shift = np.array([wy1, wx1, wy1, wx1])
    wh, ww = wy2 - wy1, wx2 - wx1
    scale = np.array([wh, ww, wh, ww])
    boxes = np.divide(boxes - shift, scale)
    boxes = denorm_boxes(boxes, original_image_shape[:2])
    exclude_ix = np.where((boxes[:, 2] - boxes[:, 0]) * (boxes[:, 3] - boxes[:, 1]) <= 0)[0]
    if exclude_ix.shape[0] > 0:
        boxes = np.delete(boxes, exclude_ix, axis=0)
        class_ids = np.delete(class_ids, exclude_ix, axis=0)
        scores = np.delete(scores, exclude_ix, axis=0)
    return boxes, class_ids, scores


# -------------------------------------------------------------------- Faster R-CNN
FRCNN_BASE_ANCHORS = np.array([[-84., -40., 99., 55.], [-176., -88., 191., 103.], [-360., -184., 375., 199.],
                               [-56., -56., 71., 71.], [-120., -120., 135., 135.], [-248., -248., 263., 263.],
                               [-36., -80., 51., 95.], [-80., -168., 95., 183.], [-168., -344., 183., 359.]])


def frcnn_decode(anchors, deltas):
    anchors, deltas = _f64(anchors), _f64(deltas)
    out = np.empty_like(deltas)
    lib().orc_frcnn_decode(_p(anchors), _p(deltas), c_int64(anchors.shape[0]), _p(out))
    return out


def frcnn_nms_sorted(boxes, thr: float, max_out: int):
    boxes = _f64(boxes)
    keep = np.empty(max(max_out, 1), np.int32)
    cnt = lib().orc_frcnn_nms_sorted(_p(boxes), c_int32(boxes.shape[0]), c_double(thr), c_int32(max_out), _p(keep))
    return keep[:cnt].copy()


def frcnn_proposals(probs, bbox, image_h: int, image_w: int, pre_n: int, post_n: int, thr: float,
                    min_hw: int = 16, feat_stride: int = 16, base_anchors=FRCNN_BASE_ANCHORS):
    """FasterRCNN Proposals.build with the intended top-N. Returns [n,5] float32."""
    probs, bbox = _f64(probs), _f64(bbox)
    _, h, w, c = probs.shape
    na = c // 2
    base = _f64(base_anchors)
    out = np.empty((post_n, 5), np.float32)
    cnt = lib().orc_frcnn_proposals(_p(probs), _p(bbox), c_int32(h), c_int32(w), c_int32(na), _p(base),
                                    c_int32(feat_stride), c_int32(image_h), c_int32(image_w), c_int32(min_hw),
                                    c_int32(pre_n), c_int32(post_n), c_double(thr), _p(out))
    return out[:cnt].copy()


def roi_pool(feature_map, proposals, image_h: float, image_w: float):
    feature_map, proposals = _f32(feature_map), _f32(proposals).reshape(-1, 5)
    B, H, W, D = feature_map.shape
    n = proposals.shape[0]
    out = np.empty((n, 7, 7, D), np.float32)
    lib().orc_roi_pool(_p(feature_map), c_int32(B), c_int32(H), c_int32(W), c_int32(D), _p(proposals), c_int32(n),
                       c_float(image_h), c_float(image_w), _p(out))
    return out
