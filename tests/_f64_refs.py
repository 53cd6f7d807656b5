"""Float64 restatements of the outputs that no reference-run golden pins: the mask targets of DetectionTargetLayer and
the forward values of the four head losses. They are written from the text of the models, not from the kernels or the
oracle, so that an error shared by ``csrc/`` and ``oracle/`` shows up as a disagreement with them.

Each reference keeps only the fp32 semantics the contract fixes (clip constants, the first-max argmax, overflow to
inf / NaN where the reference's fp32 graph overflows) and otherwise computes in float64. Instead of a tolerance, each
result comes with the set of pixels it can decide (mask targets) or an error budget derived from the fp32 formula
(losses)."""
import numpy as np

U = 2.0 ** -24                       # unit roundoff of fp32
F32_MAX = float(np.finfo(np.float32).max)
EPS32 = float(np.float32(1e-7))                          # K.epsilon() as the fp32 graph holds it
HI32 = float(np.float32(1.0) - np.float32(1e-7))         # 1 - epsilon, rounded in fp32


def _f32_exact(*xs):
    """Elementwise: every array is made of fp32 numbers (so fp32 arithmetic that lands on them is exact)."""
    ok = True
    with np.errstate(all="ignore"):
        for x in xs:
            x = np.asarray(x, np.float64)
            ok = ok & (np.isfinite(x) & (x.astype(np.float32).astype(np.float64) == x))
    return ok


# ------------------------------------------------------------------ crop_and_resize
def crop_and_resize_f64(image, boxes, box_ind, ph, pw, extrapolation=0.0, edge_tol=1e-4):
    """tf.image.crop_and_resize (bilinear) in float64: in_y = y1*(H-1) + y*(y2-y1)*(H-1)/(ph-1) (the centre
    0.5*(y1+y2)*(H-1) when ph == 1), samples outside [0, H-1] x [0, W-1] take the extrapolation value.
    Returns (crops [n,ph,pw,D] float64, comparable [n,ph,pw] bool). Not comparable: crops of an out-of-range box_ind
    (left untouched by the kernels), non-finite positions, and samples within edge_tol pixel of the feature map's edge,
    whose in/out decision rests on the fp32 rounding of the kernels' sample position."""
    img = np.asarray(image, np.float64)
    B, H, W, D = img.shape
    n = boxes.shape[0]
    out = np.zeros((n, ph, pw, D))
    ok = np.zeros((n, ph, pw), bool)

    def axis(a1, a2, size, steps):
        if steps > 1:
            pos = a1 * (size - 1) + np.arange(steps) * ((a2 - a1) * (size - 1) / (steps - 1))
        else:
            pos = np.array([0.5 * (a1 + a2) * (size - 1)])
        fin = np.isfinite(pos)
        p = np.where(fin, pos, -1.0)
        inside = (p >= 0) & (p <= size - 1)
        far = fin & (np.abs(p) > edge_tol) & (np.abs(p - (size - 1)) > edge_tol)
        p = np.clip(p, 0, size - 1)
        lo = np.floor(p).astype(np.int64)
        return lo, np.ceil(p).astype(np.int64), p - lo, inside, far

    for i in range(n):
        b = int(box_ind[i])
        if not 0 <= b < B:
            continue
        y1, x1, y2, x2 = (float(v) for v in boxes[i])
        with np.errstate(invalid="ignore"):
            top, bot, yl, in_y, far_y = axis(y1, y2, H, ph)
            left, right, xl, in_x, far_x = axis(x1, x2, W, pw)
        f = img[b]
        xl_, yl_ = xl[None, :, None], yl[:, None, None]
        t = f[top][:, left] + (f[top][:, right] - f[top][:, left]) * xl_
        bt = f[bot][:, left] + (f[bot][:, right] - f[bot][:, left]) * xl_
        v = t + (bt - t) * yl_
        out[i] = np.where((in_y[:, None] & in_x[None, :])[..., None], v, extrapolation)
        ok[i] = far_y[:, None] & far_x[None, :]
    return out, ok


# ------------------------------------------------------------------ mask targets
def _sample_axis(a1, a2, size, steps):
    """Sample positions of one crop_and_resize axis, whether each is exactly what fp32 arithmetic gives, and how far
    (in pixels) an fp32 evaluation of the same formula can be from it: a few ulps of |box| * (size - 1), 16 ulps
    taken, plus 1e-4 px."""
    with np.errstate(all="ignore"):
        if steps > 1:
            scale, span = a1 * (size - 1), (a2 - a1) * (size - 1)
            step = span / (steps - 1)
            k = np.arange(steps, dtype=np.float64)
            pos = scale + k * step
            exact = _f32_exact(a1, a2, scale, a2 - a1, span, step, k * step, pos) & (step * (steps - 1) == span)
        else:
            pos = np.array([0.5 * (a1 + a2) * (size - 1)])
            exact = _f32_exact(a1, a2, a1 + a2, pos)
        tol = 1e-4 + 16 * U * (abs(a1) + abs(a2) + 1) * (size - 1)
    if not np.isfinite(tol):                  # every position is inf or NaN: no sample is near the bounds
        tol = 0.0
    return pos, np.broadcast_to(exact, pos.shape), tol


def mask_targets_f64(rois, gt_boxes, gt_rows, gt_masks, mask_shape, use_mini_mask, hwg_layout=True):
    """Mask targets of one image's positive ROIs, restated from matterport Mask_RCNN ``detection_targets_graph``
    (mrcnn/model.py): with mini masks the ROI is re-expressed in its GT box's frame,
    ``boxes = (roi - gt.y1x1y1x1) / (gt_h, gt_w, gt_h, gt_w)``; then ``masks = crop_and_resize(gt_mask, boxes,
    MASK_SHAPE)`` (bilinear, extrapolation 0) and ``tf.round`` (half to even).

    rois [P,4], gt_boxes [G,4], gt_rows [P] (GT row of each ROI, in the uncompacted GT list), gt_masks [Mh,Mw,G]
    (hwg_layout) or [G,Mh,Mw]. Returns (value [P,mh,mw] float64 before rounding, decidable [P,mh,mw] bool); the target
    is ``np.round(value)`` where decidable. A pixel is not decidable when its value is within the fp32 position error
    of 0.5, or when a sample lies within that error of the mask's [0, M-1] bounds and the pixel could round to 1 had
    it fallen inside; away from both, bilinear interpolation is continuous and fp32 rounding cannot change the result.
    A pixel whose every intermediate is an fp32 number (exact ties such as 0.5 from 0/1 masks at half-pixel taps) is
    decidable: fp32 arithmetic reproduces it exactly."""
    rois, gt_boxes = np.asarray(rois, np.float64), np.asarray(gt_boxes, np.float64)
    masks = np.asarray(gt_masks, np.float64)
    if hwg_layout:
        masks = masks.transpose(2, 0, 1)
    _, Mh, Mw = masks.shape
    mh, mw = mask_shape
    P = rois.shape[0]
    value = np.zeros((P, mh, mw))
    decidable = np.zeros((P, mh, mw), bool)
    for i in range(P):
        g = int(gt_rows[i])
        box = rois[i]
        if use_mini_mask:
            gt = gt_boxes[g]
            gh, gw = gt[2] - gt[0], gt[3] - gt[1]
            with np.errstate(all="ignore"):
                box = (box - gt[[0, 1, 0, 1]]) / np.array([gh, gw, gh, gw])
        py, ey, ty = _sample_axis(box[0], box[2], Mh, mh)
        px, ex, tx = _sample_axis(box[1], box[3], Mw, mw)
        f = masks[g]
        axes = []
        for pos, exact, size, tol in ((py, ey, Mh, ty), (px, ex, Mw, tx)):
            fin = np.isfinite(pos)
            p = np.where(fin, pos, -1.0)
            inside = (p >= 0) & (p <= size - 1)
            near = fin & ~exact & ((np.abs(p) <= tol) | (np.abs(p - (size - 1)) <= tol))
            p = np.clip(p, 0, size - 1)
            lo = np.floor(p)
            axes.append((lo.astype(np.int64), np.ceil(p).astype(np.int64), p - lo, inside, near))
        (top, bot, yl, in_y, near_y), (left, right, xl, in_x, near_x) = axes
        tl, tr = f[top][:, left], f[top][:, right]
        bl, br = f[bot][:, left], f[bot][:, right]
        xl_, yl_ = xl[None, :], yl[:, None]
        t = tl + (tr - tl) * xl_
        bt = bl + (br - bl) * xl_
        v_in = t + (bt - t) * yl_                            # the value had every sample fallen inside
        v = np.where(in_y[:, None] & in_x[None, :], v_in, 0.0)
        # |d value / d position| <= 1 px^-1 per axis for mask values in [0, 1]; 1e-6 covers the fp32 lerp itself
        vtol = 2 * max(ty, tx) + 1e-6
        edge = (near_y[:, None] | near_x[None, :]) & (np.abs(v_in) >= 0.5 - vtol)
        ok = ~(np.abs(v - 0.5) <= vtol) & ~edge
        exact = (ey[:, None] & ex[None, :] &
                 _f32_exact(tl, tr, bl, br, tr - tl, (tr - tl) * xl_, t, br - bl, (br - bl) * xl_, bt, bt - t,
                            (bt - t) * yl_, v_in))
        value[i], decidable[i] = v, ok | exact
    return value, decidable


def gt_assignment_f64(rois, gt_boxes, gt_class_ids):
    """GT box of every ROI as data_processor.py:576-579,:610 choose it: get_iou_tf (no +1, no canonicalisation) over
    the GT boxes with a non-zero class, first maximum (a NaN IoU never wins). Returns (row in the uncompacted GT list,
    index in the compacted list, ambiguous) where ambiguous marks ROIs whose two best IoUs are within 1e-6."""
    r, g = np.asarray(rois, np.float64), np.asarray(gt_boxes, np.float64)
    valid = np.nonzero(np.asarray(gt_class_ids) != 0)[0]
    g = g[valid]
    with np.errstate(all="ignore"):
        p_area = ((r[:, 2] - r[:, 0]) * (r[:, 3] - r[:, 1]))[:, None]
        g_area = ((g[:, 2] - g[:, 0]) * (g[:, 3] - g[:, 1]))[None, :]
        ih = np.maximum(np.minimum(r[:, None, 2], g[None, :, 2]) - np.maximum(r[:, None, 0], g[None, :, 0]), 0)
        iw = np.maximum(np.minimum(r[:, None, 3], g[None, :, 3]) - np.maximum(r[:, None, 1], g[None, :, 1]), 0)
        inter = ih * iw
        iou = inter / (p_area + g_area - inter)
    iou = np.where(np.isnan(iou), -np.inf, iou)
    arg = iou.argmax(1) if valid.size else np.zeros(r.shape[0], np.int64)
    if valid.size > 1:
        top2 = -np.sort(-iou, axis=1)[:, :2]
        ambiguous = top2[:, 0] - top2[:, 1] <= 1e-6
    else:
        ambiguous = np.zeros(r.shape[0], bool)
    return (valid[arg] if valid.size else arg), arg, ambiguous


# ------------------------------------------------------------------ head losses
def first_max(x):
    """tf.argmax over the last axis as a serial scan with a strict '>': the first maximum wins and a NaN never
    replaces the running maximum (a NaN at index 0 stays). Returns (argmax, running maximum)."""
    x = np.asarray(x)
    arg = np.zeros(x.shape[:-1], np.int64)
    m = x[..., 0].copy()
    for j in range(1, x.shape[-1]):
        up = x[..., j] > m
        arg[up] = j
        m[up] = x[..., j][up]
    return arg, m


def _softmax_ce(x, label):
    """Sparse softmax cross-entropy of rows x [n,C] (float64 of fp32 logits) at integer labels, with its fp32 error
    bound. The kernels evaluate log(sum_j exp(x_j - m)) - (x_label - m) in fp32, m the running maximum. Rounding
    x_j - m, exp, the C-term serial sum and log put at most (C + 1) u on log(s) for s >= 1, plus u |log s|; x_label - m
    and the final subtraction add u |x_label - m| and u (|log s| + |x_label - m|). So the error is at most
    c u (|log s| + |x_label - m| + 1) with c = C + 2 (4 for the RPN's two classes)."""
    n, C = x.shape
    _, m = first_max(x)
    with np.errstate(all="ignore"):
        gap = x[np.arange(n), label] - m
        s = np.exp(x - m[:, None]).sum(1)
        ls = np.log(s)
        ce = ls - gap
        # an fp32 gap beyond the fp32 range is -inf there: the loss is +inf (a NaN from inf - inf stays NaN)
        over = np.isfinite(gap) & np.isinf(gap.astype(np.float32))
        ce = np.where(over & ~np.isnan(ce), np.inf, ce)
        bound = (C + 2) * U * (np.abs(ls) + np.abs(gap) + 1)
    return ce, bound


def _mean(terms, bounds, count):
    """(mean, budget): the sum of the per-term bounds over the count, the fp64 accumulation (count * 2^-53 of the sum
    of |terms|) and the final rounding to fp32 (u |L|)."""
    if count == 0:
        return 0.0, 0.0
    with np.errstate(all="ignore"):
        L = float(np.sum(terms) / count)
        budget = float(np.sum(bounds) / count + count * 2.0 ** -53 * np.sum(np.abs(terms)) / count + U * abs(L))
    return L, budget


def smooth_l1_f64(target, pred):
    """loss_optimize.py:79-81 per element: 0.5 d^2 when d = |target - pred| < 1, d - 0.5 otherwise. The fp32 graph
    evaluates (0.5 * less) * (d * d) + (d - 0.5) * (1 - less) on every element: where d * d overflows fp32, 0 * inf
    makes the element NaN. Error bound of the fp32 evaluation: d, d * d and d - 0.5 are each rounded once, at most
    3 u (|d| + 0.5 + 1)."""
    t, p = np.asarray(target, np.float64), np.asarray(pred, np.float64)
    with np.errstate(all="ignore"):
        d = np.abs(t - p)
        l = np.where(d < 1, 0.5 * d * d, d - 0.5)
        d32 = d.astype(np.float32).astype(np.float64)
        l = np.where(np.isinf((d32 * d32).astype(np.float32)) | np.isnan(d), np.nan, l)
        bound = 3 * U * (d + 0.5 + 1)
    return l, bound


def rpn_losses_f64(rpn_target_class, rpn_class_logits, rpn_target_bbox, rpn_pred_box):
    """Loss.rpn_class_loss (loss_optimize.py:11-44) and Loss.rpn_box_loss (:47-87): anchors with a non-zero target
    (not_equal(0)) enter the cross-entropy with label equal(target, 1); the positives (equal 1) of image b, in anchor
    order, pair with the first rows of rpn_target_bbox[b], at most T of them; means, 0 when empty.
    Returns (class_loss, class_budget, box_loss, box_budget, rpn_pred_box_pos)."""
    lg = np.asarray(rpn_class_logits, np.float64)
    B, A = lg.shape[:2]
    tc = np.asarray(rpn_target_class).reshape(B, A)
    sel = tc != 0
    ce, cb = _softmax_ce(lg[sel], (tc[sel] == 1).astype(np.int64))
    cls = _mean(ce, cb, ce.size)
    tb, pb = np.asarray(rpn_target_bbox, np.float64), np.asarray(rpn_pred_box, np.float64)
    pos = tc == 1
    T = tb.shape[1]
    pairs = [(tb[b, :min(int(pos[b].sum()), T)], pb[b][pos[b]][:T]) for b in range(B)]
    t = np.concatenate([q[0] for q in pairs]).reshape(-1)
    p = np.concatenate([q[1] for q in pairs]).reshape(-1)
    l, lb = smooth_l1_f64(t, p)
    box = _mean(l, lb, l.size)
    return cls[0], cls[1], box[0], box[1], pb[pos].astype(np.float32)


def bce_f64(target, pred):
    """K.binary_crossentropy(target, output) (Keras 2, TF backend) per element: o = clip(output, eps, 1 - eps) with the
    fp32 constants, z = log(o / (1 - o)), then sigmoid_cross_entropy_with_logits = max(z, 0) - z t + log1p(exp(-|z|)).
    Error bound of the fp32 evaluation: z carries u (3 + |z|) (1 - o, the quotient, log), which the loss multiplies by
    at most 1.5 + |t|; z t, the subtraction and the final addition add one rounding each. With |t| <= (|t| + 2) and
    3 + |z| <= 3 (|z| + 1) that is at most 8 u (|z| + 1)(|t| + 2)."""
    t, p = np.asarray(target, np.float64), np.asarray(pred, np.float64)
    with np.errstate(all="ignore"):
        o = np.minimum(np.maximum(p, EPS32), HI32)
        o = np.where(np.isnan(p), np.nan, o)
        z = np.log(o / (1 - o))
        l = (np.maximum(z, 0) - z * t) + np.log1p(np.exp(-np.abs(z)))
        bound = 8 * U * (np.abs(z) + 1) * (np.abs(t) + 2)
    return l, bound


def mrcnn_losses_f64(mrcnn_target_class_ids, mrcnn_pred_logits, batch_active_class_ids, mrcnn_target_box,
                     mrcnn_pred_box):
    """Loss.mrcnn_class_loss (loss_optimize.py:89-151) and Loss.mrcnn_box_loss (:154-201) for labels in [0, C):
    pred_active = batch_active_class_ids[0][argmax(logits)]; class loss = sum(ce * pred_active) / sum(pred_active)
    (NaN when no predicted class is active); box loss = mean BCE of the target class's predicted box over the ROIs with
    a positive label, 0 when there are none. Returns (pred_active, class_loss, class_budget, box_loss, box_budget)."""
    ids = np.asarray(mrcnn_target_class_ids).astype(np.int64)
    lg = np.asarray(mrcnn_pred_logits, np.float64)
    act = np.asarray(batch_active_class_ids, np.float64)
    B, R, C = lg.shape
    assert ((ids >= 0) & (ids < C)).all(), "labels outside [0, C) are outside the reference's domain"
    arg, _ = first_max(lg.reshape(-1, C))
    pa = act[0][arg]
    ce, cb = _softmax_ce(lg.reshape(-1, C), ids.reshape(-1))
    with np.errstate(all="ignore"):
        w = ce * pa
        den = float(pa.sum())
        num = float(w.sum())
        cls = num / den if den != 0 else np.nan
        cbud = (float(np.sum(np.abs(pa) * (cb + U * np.abs(ce)))) + 2.0 ** -53 * len(w) * float(np.sum(np.abs(w))))
        cbud = cbud / abs(den) + U * abs(cls) if den != 0 else np.nan
    posm = ids > 0
    t = np.asarray(mrcnn_target_box, np.float64)[posm]
    p = np.asarray(mrcnn_pred_box, np.float64)[posm, ids[posm]]
    l, lb = bce_f64(t, p)
    box = _mean(l, lb, l.size)
    return pa.reshape(B, R).astype(np.float32), cls, cbud, box[0], box[1]


def assert_loss(got, want, budget, what=""):
    """got (fp32) against a float64 reference value: within the budget where the reference is finite, the same inf or
    NaN where the fp32 graph overflows."""
    got = float(got)
    if np.isnan(want):
        assert np.isnan(got), f"{what}: got {got!r}, want NaN"
    elif np.isinf(want) or abs(want) > F32_MAX:
        assert got == np.copysign(np.inf, want), f"{what}: got {got!r}, want {want!r} (inf in fp32)"
    else:
        assert abs(got - want) <= budget, f"{what}: got {got!r}, want {want!r}, |err| {abs(got - want):.3e} > {budget:.3e}"
