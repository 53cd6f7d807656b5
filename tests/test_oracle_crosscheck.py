"""The two independent CPU restatements (C: oracle/odhead_oracle.c, numpy: oracle/np_layers.py) must agree
bit for bit, on the reference's own debug() input recipes (seed + shape) and on hand-built edge cases.
Also cross-checks NMS against torchvision where the semantics coincide."""
import numpy as np
import pytest

import oracle
from oracle import np_layers as npl
from objectdetection_b200.config import config as Conf, ShapesConfig

f32 = np.float32


def bits(a):
    return np.ascontiguousarray(a, f32).view(np.uint32)


def assert_bits_equal(a, b, what=""):
    a, b = np.asarray(a, f32), np.asarray(b, f32)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    same = (bits(a) == bits(b)) | (np.isnan(a) & np.isnan(b))
    assert same.all(), f"{what}: {np.argwhere(~same)[:5]}"


# ------------------------------------------------------------------ top-k
def test_topk_ties_and_strides():
    rs = np.random.RandomState(0)
    s = (rs.randint(0, 50, size=(3, 500)) / 50).astype(f32)       # many ties
    s[0, 7] = -0.0
    s[0, 9] = 0.0
    v, i = oracle.topk(s, 200)
    v2, i2 = npl.tf_top_k(s, 200)
    assert np.array_equal(i, i2) and np.array_equal(v, v2)
    probs = rs.random_sample((2, 300, 2)).astype(f32)
    v, i = oracle.topk(probs[:, :, 1], 300)                         # strided view, k == A
    v2, i2 = npl.tf_top_k(probs[:, :, 1], 300)
    assert np.array_equal(i, i2) and np.array_equal(v, v2)
    assert np.all(np.diff(v, axis=1) <= 0)


# ------------------------------------------------------------------ NMS
def _random_boxes(rs, n, scale=1.0, flip=False):
    yx = rs.random_sample((n, 2)) * 0.8
    hw = rs.random_sample((n, 2)) * 0.3 + 0.01
    b = np.concatenate([yx, yx + hw], axis=1) * scale
    if flip:
        sw = rs.random_sample(n) < 0.3
        b[sw] = b[sw][:, [2, 3, 0, 1]]
    return b.astype(f32)


@pytest.mark.parametrize("thr", [0.3, 0.5, 0.7])
def test_nms_c_vs_numpy(thr):
    rs = np.random.RandomState(int(thr * 10))
    boxes = _random_boxes(rs, 300, flip=True)
    boxes[5] = boxes[6]                              # duplicates
    boxes[10, 2:] = boxes[10, :2]                    # zero area
    scores = (rs.randint(0, 40, 300) / 40).astype(f32)   # ties
    for max_out in (5, 100, 300):
        assert np.array_equal(oracle.nms(boxes, scores, max_out, thr),
                              npl.tf_non_max_suppression(boxes, scores, max_out, thr))


def test_nms_vs_torchvision():
    torch = pytest.importorskip("torch")
    tv = pytest.importorskip("torchvision")
    rs = np.random.RandomState(3)
    boxes = _random_boxes(rs, 500, scale=100.0)
    scores = rs.permutation(500).astype(f32)
    for thr in (0.3, 0.5, 0.7):
        keep = oracle.nms(boxes, scores, 500, thr)
        # torchvision boxes are (x1,y1,x2,y2); IoU is symmetric in the axis naming
        tvk = tv.ops.nms(torch.from_numpy(boxes[:, [1, 0, 3, 2]]), torch.from_numpy(scores), thr).numpy()
        assert np.array_equal(keep, tvk)


def test_nms_zero_area_never_suppresses():
    boxes = np.array([[0, 0, 1, 1], [0.5, 0.5, 0.5, 0.5], [0, 0, 1, 1], [0.2, 0.2, 0.2, 0.9]], f32)
    scores = np.array([0.9, 0.8, 0.7, 0.6], f32)
    assert oracle.nms(boxes, scores, 10, 0.1).tolist() == [0, 1, 3]


# ------------------------------------------------------------------ decode / clip
def test_decode_clip_c_vs_numpy():
    rs = np.random.RandomState(1)
    a = rs.random_sample((2, 257, 4)).astype(f32)
    d = rs.normal(0, 1, size=(2, 257, 4)).astype(f32)
    dec = oracle.apply_box_deltas(a, d)
    assert_bits_equal(dec, npl.apply_box_deltas(a, d), "decode")
    assert_bits_equal(oracle.clip_boxes(dec, np.array([0, 0, 1, 1], f32)),
                      npl.clip_boxes_to_01(dec, np.array([0, 0, 1, 1], f32)), "clip")
    win = np.array([[0.1, 0.2, 0.8, 0.9], [0, 0.3, 1, 0.7]], f32)
    ref = np.stack([npl.clip_boxes_to_01(dec[b], win[b]) for b in range(2)])
    assert_bits_equal(oracle.clip_boxes(dec, win), ref, "clip per image")


# ------------------------------------------------------------------ crop_and_resize / roi align
def test_crop_and_resize_c_vs_numpy_edges():
    rs = np.random.RandomState(2)
    img = rs.random_sample((2, 9, 11, 8)).astype(f32)
    boxes = np.array([[0, 0, 1, 1], [0.1, 0.2, 0.7, 0.9], [0.3, 0.3, 0.3, 0.3], [-0.2, -0.1, 0.5, 0.5],
                      [0.5, 0.5, 1.3, 1.2], [0.9, 0.8, 0.1, 0.2], [0, 0, 0, 0], [0.25, 0.5, 0.75, 1.0]], f32)
    bi = np.array([0, 1, 0, 1, 0, 1, 0, 5], np.int32)                # last one: out-of-range -> skipped
    for crop in ((7, 7), (14, 14), (1, 1), (1, 3), (2, 2)):
        c = oracle.crop_and_resize(img, boxes, bi, *crop)
        n = npl.tf_crop_and_resize(img, boxes, bi, crop)
        assert_bits_equal(c, n, f"crop {crop}")
    # interior boxes coincide with align_corners bilinear grid sampling
    torch = pytest.importorskip("torch")
    b = np.array([[0.1, 0.2, 0.7, 0.9]], f32)
    ys = torch.linspace(float(b[0, 0]), float(b[0, 2]), 7) * 2 - 1
    xs = torch.linspace(float(b[0, 1]), float(b[0, 3]), 7) * 2 - 1
    grid = torch.stack(torch.meshgrid(ys, xs, indexing="ij")[::-1], dim=-1)[None]
    ref = torch.nn.functional.grid_sample(torch.from_numpy(img[:1]).permute(0, 3, 1, 2), grid, mode="bilinear",
                                          align_corners=True).permute(0, 2, 3, 1).numpy()
    got = oracle.crop_and_resize(img, b, np.array([0], np.int32), 7, 7)
    assert np.allclose(got, ref, rtol=1e-4, atol=1e-5)


def test_roi_pooling_debug_recipe():
    """maskrcnn.py:327-345 recipe (seed 255) at a reduced pyramid so the numpy loops finish quickly."""
    np.random.seed(255)
    nb, D = 2, 8
    fmaps = [np.array(np.random.random((nb, s, s, D)), dtype="float32") for s in (64, 32, 16, 8)]
    props = np.array(np.random.random((nb, 60, 4)), dtype="float32")
    props[1, 50:] = 0                                     # zero padded rows
    props[0, 3] = [0.4, 0.4, 0.4001, 0.4001]              # tiny -> level 2
    props[0, 4] = [0.0, 0.0, 1.0, 1.0]                    # full 256 px image -> level 4
    for pool in ([7, 7], [14, 14]):
        c, clv = oracle.pyramid_roi_align(fmaps, props, 256, 256, pool[0], pool[1])
        n, nlv = npl.roi_pooling([256, 256], pool, [2, 3, 4, 5], props, fmaps)
        assert np.array_equal(clv, nlv)
        assert set(np.unique(clv)) <= {2, 3, 4, 5} and len(np.unique(clv)) >= 3
        assert_bits_equal(c, n, f"pooled {pool}")
    assert clv[1, 55] == 2 and clv[0, 4] == 4 and clv[0, 3] == 2


def test_roi_level_degenerate():
    rois = np.array([[0, 0, 0, 0], [0.5, 0.5, 0.2, 0.9], [np.nan, 0, 1, 1], [0, 0, np.inf, 1]], f32)
    assert oracle.roi_level(rois, 1024, 1024).tolist() == [2, 2, 2, 2]
    # 224 px square at 1024 -> level 4; half-integer boundary rounds to even
    s = 224 / 1024
    assert oracle.roi_level(np.array([[0, 0, s, s]], f32), 1024, 1024).tolist() == [4]
    assert oracle.roi_level(np.array([[0, 0, 2 * s, 2 * s]], f32), 1024, 1024).tolist() == [5]


# ------------------------------------------------------------------ ProposalLayer
def test_proposals_debug_recipe():
    """proposals_tf.py:331-345 recipe: seed 325, (1,4092,{2,4,4}) uniform inputs."""
    np.random.seed(325)
    probs = np.array(np.random.random((1, 4092, 2)), dtype="float32")
    bbox = np.array(np.random.random((1, 4092, 4)), dtype="float32")
    anchors = np.array(np.random.random((1, 4092, 4)), dtype="float32")
    conf = Conf()
    out, dbg = oracle.proposal_forward(probs, bbox, anchors, conf.RPN_BBOX_STDDEV, conf.PRE_NMS_ROIS_COUNT,
                                       conf.POST_NMS_ROIS_INFERENCE, conf.RPN_NMS_THRESHOLD, debug=True)
    ref, rdbg = npl.proposals(conf, probs, bbox, anchors)
    assert np.array_equal(dbg["ix"], rdbg["ix"])
    for k in ("scores", "bbox_delta", "anchors", "anchor_delta", "anchor_delta_clipped"):
        assert_bits_equal(dbg[k], rdbg[k], k)
    n = int(dbg["num_kept"][0])
    assert np.array_equal(dbg["keep_idx"][0, :n], rdbg["keep_idx"][0]) and np.all(dbg["keep_idx"][0, n:] == -1)
    assert_bits_equal(out, ref, "proposals")
    assert out.shape == (1, 1000, 4)


def test_proposals_realistic_batch_with_padding():
    rs = np.random.RandomState(5)
    conf = ShapesConfig()
    shapes = oracle.get_resnet_stage_shapes(conf.RESNET_STRIDES, conf.IMAGE_SHAPE)
    anchors = oracle.gen_anchors(conf.IMAGE_SHAPE, 3, conf.RPN_ANCHOR_SCALES, conf.RPN_ANCHOR_RATIOS, shapes,
                                 conf.RESNET_STRIDES, conf.RPN_ANCHOR_STRIDE)
    A = anchors.shape[1]
    fg = rs.beta(0.5, 4, size=(3, A)).astype(f32)
    probs = np.stack([1 - fg, fg], axis=2).astype(f32)
    bbox = rs.normal(0, 1, size=(3, A, 4)).astype(f32)
    conf.RPN_NMS_THRESHOLD = 0.1                          # forces < N survivors -> zero padded rows
    conf.PRE_NMS_ROIS_COUNT, conf.POST_NMS_ROIS_INFERENCE = 700, 400
    out = oracle.proposal_forward(probs, bbox, anchors, conf.RPN_BBOX_STDDEV, conf.PRE_NMS_ROIS_COUNT,
                                  conf.POST_NMS_ROIS_INFERENCE, conf.RPN_NMS_THRESHOLD)
    ref, _ = npl.proposals(conf, probs, bbox, anchors)
    assert_bits_equal(out, ref, "proposals")
    assert (np.abs(out).sum(axis=2) == 0).any()


# ------------------------------------------------------------------ DetectionTargetLayer
def _target_case(rs, N, G, n_valid_gt, n_pad):
    props = _random_boxes(rs, N)
    gt = np.zeros((G, 4), f32)
    cls = np.zeros(G, np.int32)
    src = rs.choice(N - n_pad, n_valid_gt, replace=False)
    gt[:n_valid_gt] = props[src] + rs.normal(0, 0.01, size=(n_valid_gt, 4)).astype(f32)
    cls[:n_valid_gt] = rs.randint(1, 81, n_valid_gt)
    props[N - n_pad:] = 0
    return props, cls, gt, rs.permutation(N).astype(np.int32), rs.permutation(N).astype(np.int32)


@pytest.mark.parametrize("N,G,nv,pad,conf_cls", [(200, 20, 7, 30, Conf), (120, 10, 3, 0, ShapesConfig),
                                                 (64, 8, 0, 10, ShapesConfig), (300, 100, 100, 100, Conf)])
def test_detection_targets_c_vs_numpy(N, G, nv, pad, conf_cls):
    rs = np.random.RandomState(N + G)
    conf = conf_cls()
    props, cls, gt, pp, pn = _target_case(rs, N, G, nv, pad)
    rois, rcls, deltas, dbg = oracle.detection_targets(props, cls, gt, pp, pn, conf.MRCNN_TRAIN_ROIS_PER_IMAGE,
                                                       conf.BBOX_STD_DEV)
    r_rois, r_cls, r_deltas, rdbg = npl.build_detection_target(conf, props, cls, gt, pp, pn)
    n_prop, n_gt, n_pos, n_neg, pos_count, neg_count = dbg["counts"]
    assert (n_prop, n_gt) == (N - pad, nv)
    assert np.array_equal(dbg["pos_indices"][:n_pos], rdbg["pos_all"]) and np.all(dbg["pos_indices"][n_pos:] == -1)
    assert np.array_equal(dbg["neg_indices"][:n_neg], rdbg["neg_all"])
    assert pos_count == rdbg["pos_count"] and neg_count == len(rdbg["neg_indices"])
    assert np.array_equal(dbg["sampled_pos"][:pos_count], rdbg["pos_indices"])
    assert np.array_equal(dbg["sampled_neg"][:neg_count], rdbg["neg_indices"])
    assert np.array_equal(dbg["gt_assignment"][:pos_count], rdbg["assign"])
    assert_bits_equal(dbg["iou"][:n_prop, :n_gt], rdbg["iou"], "iou")
    assert_bits_equal(rois, r_rois, "rois")
    assert np.array_equal(rcls, r_cls)
    assert_bits_equal(deltas, r_deltas, "deltas")
    if nv > 0:
        assert pos_count > 0 and rcls[0, :pos_count].min() >= 1
    assert rois.shape == (conf.MRCNN_TRAIN_ROIS_PER_IMAGE, 4) and rcls.shape == (1, conf.MRCNN_TRAIN_ROIS_PER_IMAGE)


def test_detection_target_counts_fit_for_all_R():
    """pos_count + neg_count never exceeds R for the fp32 count arithmetic of data_processor.py:586-594."""
    inv = f32(1 / 0.33)
    for R in range(1, 2049):
        p = int(R * 0.33)
        assert int(inv * f32(p)) - p + p <= R, R
    assert int(inv * f32(66)) - 66 == 134 and int(inv * f32(10)) - 10 == 20


# ------------------------------------------------------------------ DetectionLayer
def test_detection_debug_recipe():
    """detection.py:285-310 recipe: seed 863, (1,8,4) proposals/probs, (1,8,4,4) deltas, window [131,0,893,1024]."""
    np.random.seed(863)
    props = np.array(np.random.random((1, 8, 4)), dtype="float32")
    probs = np.array(np.random.random((1, 8, 4)), dtype="float32")
    bbox = np.array(np.random.random((1, 8, 4, 4)), dtype="float32")
    win = oracle.norm_boxes(np.array([[131, 0, 893, 1024]], "int32"), (1024, 1024))
    conf = Conf()
    det = oracle.detection_forward(props, probs, bbox, win, conf.BBOX_STD_DEV, conf.DETECTION_MIN_THRESHOLD,
                                   conf.DETECTION_NMS_THRESHOLD, conf.DETECTION_POST_NMS_INSTANCES)
    ref = npl.detection_layer(conf, win, props, probs, bbox)
    assert det.shape == (1, 100, 6)
    assert_bits_equal(det, ref, "detections")
    assert (det[0, :, 4] > 0).sum() >= 1


def test_detection_many_classes_ties_and_caps():
    rs = np.random.RandomState(9)
    B, N, C = 2, 400, 6
    props = _random_boxes(rs, B * N).reshape(B, N, 4)
    logits = rs.normal(0, 1, size=(B, N, C))
    boost = rs.randint(0, C, size=(B, N))
    logits[np.arange(B)[:, None], np.arange(N)[None], boost] += 6
    probs = np.exp(logits) / np.exp(logits).sum(-1, keepdims=True)
    probs = (np.round(probs * 64) / 64).astype(f32)       # quantised -> many score ties
    bbox = rs.normal(0, 0.5, size=(B, N, C, 4)).astype(f32)
    win = np.array([[0.1, 0.0, 0.9, 1.0], [0, 0, 1, 1]], f32)
    conf = Conf()
    conf.DETECTION_POST_NMS_INSTANCES = 40                # cap binds
    det, dbg = oracle.detection_forward(props, probs, bbox, win, conf.BBOX_STD_DEV, conf.DETECTION_MIN_THRESHOLD,
                                        conf.DETECTION_NMS_THRESHOLD, 40, debug=True)
    ref = npl.detection_layer(conf, win, props, probs, bbox)
    assert_bits_equal(det, ref, "detections")
    assert dbg["nms_keep_mask"].sum(axis=1).min() > 40
    assert np.all(np.diff(det[:, :, 5], axis=1) <= 0)
    empty = oracle.detection_forward(props, np.full_like(probs, 1.0 / C), bbox, win, conf.BBOX_STD_DEV, 0.7, 0.3, 40)
    assert not empty.any()


def test_unmold_detection_golden(golden):
    boxes, cls, scores = oracle.unmold_detection((600, 800, 3), (1024, 1024, 3), golden["unmold_in"],
                                                 np.array([131, 0, 893, 1024]))
    assert boxes.dtype == np.int32 and np.array_equal(boxes, golden["unmold_boxes"])
    assert np.array_equal(cls, golden["unmold_class_ids"]) and np.array_equal(scores, golden["unmold_scores"])
    assert boxes.shape[0] < 37


def test_mask_targets_oracle_properties():
    """oracle.mask_targets (parity unpinned, matterport semantics): a full-ones GT mask gives an all-ones target for a
    ROI inside the GT box; an ROI equal to the GT box reproduces the (bilinearly resampled, rounded) mini mask."""
    import oracle
    rs = np.random.RandomState(4)
    N, G, R, M = 64, 4, 32, 56
    gt = np.zeros((G, 4), np.float32)
    gt[:2] = [[0.2, 0.2, 0.6, 0.7], [0.5, 0.1, 0.9, 0.5]]
    cls = np.array([3, 7, 0, 0], np.int32)
    props = np.zeros((N, 4), np.float32)
    props[0] = gt[0]                               # IoU 1 with GT 0
    props[1] = [0.25, 0.25, 0.55, 0.65]            # inside GT 0, IoU 0.6
    props[2] = gt[1]
    props[3:40] = rs.uniform(0, 0.1, (37, 4)).astype(np.float32) + np.array([0, 0, 0.05, 0.05], np.float32)
    masks = np.zeros((M, M, G), np.float32)
    masks[:, :, 0] = 1.0
    masks[10:40, 5:30, 1] = 1.0
    perm = np.arange(N, dtype=np.int32)
    rois, rcls, deltas, dbg = oracle.detection_targets(props, cls, gt, perm, perm, R, [0.1, 0.1, 0.2, 0.2])
    assert int(dbg["counts"][4]) == 3
    t = oracle.mask_targets(rois, cls, gt, masks, dbg, (28, 28), True)
    # (an ROI equal to its GT box may lose its last row/column to fp32 rounding: in = y*55/27 can exceed 55 - TF too)
    assert t.shape == (R, 28, 28) and (t[0][:27, :27] == 1).all() and (t[1] == 1).all() and not t[3:].any()
    # ROI == GT box 1: the target is the mini mask resampled 56 -> 28 (corner aligned), rounded
    ys = np.round(np.linspace(0, M - 1, 28)).astype(int)
    coarse = masks[:, :, 1][np.ix_(ys, ys)]
    assert np.mean(t[2] == coarse) > 0.95
    full = oracle.mask_targets(rois, cls, gt, masks, dbg, (28, 28), False)
    assert full.shape == (R, 28, 28) and (full[0] == 1).all()     # ROI 0 in image coordinates lies inside the mask


def test_rpn_levels_to_flat_matches_reshape_softmax_concat():
    """oracle.rpn_levels_to_flat against an independent torch reshape/softmax/concat (rpn.py:54-66, training.py:163-166)."""
    torch = pytest.importorskip("torch")
    rs = np.random.RandomState(3)
    logits = [rs.normal(0, 3, (2, s, s, 6)).astype(f32) for s in (8, 4, 2)]
    bbox = [rs.normal(0, 1, (2, s, s, 12)).astype(f32) for s in (8, 4, 2)]
    probs, flat = oracle.rpn_levels_to_flat(logits, bbox)
    assert probs.shape == (2, 3 * (64 + 16 + 4), 2) and flat.shape == (2, 252, 4)
    want = torch.cat([torch.softmax(torch.from_numpy(c).reshape(2, -1, 2).double(), -1) for c in logits], 1).numpy()
    assert np.allclose(probs, want, rtol=5e-7, atol=1e-9)          # three fp32 roundings
    assert np.array_equal(flat, np.concatenate([d.reshape(2, -1, 4) for d in bbox], 1))
    # anchor order inside a level: y, x, anchor (the reshape of NHWC)
    assert np.array_equal(flat[1, (3 * 8 + 5) * 3 + 2], bbox[0][1, 3, 5, 8:12])


def test_head_losses_oracle_vs_torch():
    """oracle.rpn_losses / mrcnn_losses (loss_optimize.py:11-201) against independent torch float64 formulas."""
    torch = pytest.importorskip("torch")
    F = torch.nn.functional
    rs = np.random.RandomState(0)
    B, A, T = 2, 500, 16
    tc = rs.choice([-1, 0, 1], size=(B, A, 1), p=[.3, .65, .05]).astype(np.int32)
    lg = rs.normal(0, 2, (B, A, 2)).astype(f32)
    tb, pb = rs.normal(0, 1, (B, T, 4)).astype(f32), rs.normal(0, 1, (B, A, 4)).astype(f32)
    cl, bl, pos = oracle.rpn_losses(tc, lg, tb, pb)
    sel = torch.from_numpy(tc[..., 0] != 0)
    want = F.cross_entropy(torch.from_numpy(lg)[sel].double(), torch.from_numpy(tc[..., 0] == 1)[sel].long())
    assert np.isclose(cl, float(want), rtol=1e-6)
    tg, pr = [], []
    for i in range(B):
        m = tc[i, :, 0] == 1
        n = min(int(m.sum()), T)
        tg.append(tb[i, :n])
        pr.append(pb[i][m][:n])
    want = F.smooth_l1_loss(torch.from_numpy(np.concatenate(pr)).double(), torch.from_numpy(np.concatenate(tg)).double())
    assert np.isclose(bl, float(want), rtol=1e-6)
    assert np.array_equal(pos, pb[tc[..., 0] == 1])
    z = np.zeros_like(tc)
    assert oracle.rpn_losses(z, lg, tb, pb)[:2] == (0.0, 0.0)                   # K.switch(size > 0, ., 0)
    # the reference's debug() recipe for the detection-head losses (loss_optimize.py:209-219)
    R, C = 32, 4
    ids = np.zeros((2, R), np.int32)
    ids[0, 2], ids[0, 3], ids[1, 4] = 1, 2, 1
    tb2, pb2 = rs.random_sample((2, R, 4)).astype(f32), rs.random_sample((2, R, C, 4)).astype(f32)
    lg2 = rs.normal(0, 2, (2, R, C)).astype(f32)
    act = np.array([[1, 1, 0, 1], [1, 0, 0, 0]], f32)
    pa, cl2, bl2 = oracle.mrcnn_losses(ids, lg2, act, tb2, pb2)
    ce = F.cross_entropy(torch.from_numpy(lg2).double().reshape(-1, C), torch.from_numpy(ids).long().reshape(-1),
                         reduction="none").reshape(2, R)
    pa_w = torch.from_numpy(act)[0][torch.from_numpy(lg2).argmax(-1)]
    assert np.array_equal(pa, pa_w.numpy())
    assert np.isclose(cl2, float((ce * pa_w).sum() / pa_w.sum()), rtol=1e-6)
    m = ids > 0
    want = F.binary_cross_entropy(torch.from_numpy(pb2[m, ids[m]]).double(), torch.from_numpy(tb2[m]).double())
    assert np.isclose(bl2, float(want), rtol=1e-5)
    assert oracle.mrcnn_losses(np.zeros_like(ids), lg2, act, tb2, pb2)[2] == 0.0


# ------------------------------------------------------------------ the oracle's own build
def test_oracle_build_follows_the_source_bytes_not_file_times(tmp_path):
    """liboracle.so is rebuilt when the source changes, not when only its file time does (a copied tree keeps none);
    in a tree it cannot write, a stale library is built once in a temporary directory that later processes reuse."""
    import importlib.util
    import os
    import shutil
    d = tmp_path / "oracle"
    d.mkdir()
    for f in ("__init__.py", "odhead_oracle.c"):
        shutil.copy(os.path.join(os.path.dirname(oracle.__file__), f), d / f)

    def load():                     # a fresh import of the copy, as a new process would see it
        spec = importlib.util.spec_from_file_location("oracle_copy", d / "__init__.py")
        m = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(m)
        return m

    copy = load()
    lib = copy.build()
    assert lib == str(d / "liboracle.so")
    t = os.path.getmtime(lib)
    os.utime(d / "odhead_oracle.c", (t + 60, t + 60))
    assert copy.build() == lib and os.path.getmtime(lib) == t
    with open(d / "odhead_oracle.c", "a") as f:
        f.write("\n")
    assert copy.build() == lib and os.path.getmtime(lib) != t
    if os.geteuid() == 0:
        return                      # root writes into a read-only directory anyway
    with open(d / "odhead_oracle.c", "a") as f:
        f.write("\n")
    t = os.path.getmtime(lib)
    d.chmod(0o555)
    try:
        out = copy.build()
        built = os.path.getmtime(out)
        again = load()
        assert again.build() == out and again._LIB == out and os.path.getmtime(out) == built
    finally:
        d.chmod(0o755)
    assert os.path.dirname(out) != str(d) and copy._LIB == out
    assert os.path.getmtime(lib) == t
    shutil.rmtree(os.path.dirname(out))
