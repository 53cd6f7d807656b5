"""The oracle against goldens produced by the REFERENCE'S OWN layer classes.

tests/golden/reference_layers.npz was written by tests/golden/make_golden_layers.py, which imports
proposals_tf.py / maskrcnn.py / data_processor.py / detection.py / utils.py unmodified from /root/reference and runs
them through the numpy-eager TensorFlow stand-in tests/tf_shim (the three TF C++ kernels delegate to the oracle's
restatements; everything the reference itself wrote executes as written). Here — CPU only, no reference tree needed —
the C oracle (oracle/odhead_oracle.c) and the independent numpy oracle (oracle/np_layers.py) are required to equal those
files bit for bit; tests/test_gpu_parity_goldens.py asks the same of the CUDA path. A large member is stored as its
shape, a digest of all of its bits and a seeded sample of its rows (tests/golden/golden_sample.py); `bits` compares
a result with all three.
"""
import hashlib
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(HERE, "golden"))
import golden_sample  # noqa: E402
import layer_recipes as R  # noqa: E402

import oracle  # noqa: E402
from oracle import np_layers  # noqa: E402

f32 = np.float32


@pytest.fixture(scope="module")
def G():
    return golden_sample.Golden(os.path.join(HERE, "golden", "reference_layers.npz"))


def bits(a, b, what=""):
    if isinstance(b, golden_sample.Sampled):
        return b.check(a, what, bits)
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    if a.dtype.kind == "f" or b.dtype.kind == "f":
        a, b = a.astype(f32), b.astype(f32)
        same = (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))
    else:
        same = a.astype(np.int64) == b.astype(np.int64)
    if not same.all():
        bad = np.argwhere(~same)
        raise AssertionError(f"{what}: {bad.shape[0]} of {a.size} differ; first at {bad[0].tolist()}: "
                             f"got {a[tuple(bad[0])]!r} want {b[tuple(bad[0])]!r}")


def sha(a):
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), np.uint8)


def anchors_fn(conf, batch):
    shapes = oracle.get_resnet_stage_shapes(conf.RESNET_STRIDES, conf.IMAGE_SHAPE)
    return oracle.gen_anchors(conf.IMAGE_SHAPE, batch, conf.RPN_ANCHOR_SCALES, conf.RPN_ANCHOR_RATIOS, shapes,
                              conf.RESNET_STRIDES, conf.RPN_ANCHOR_STRIDE)


PROPOSAL_CASES = {"prop325": R.proposals_debug325, "proptoy": lambda: R.proposals_toy(anchors_fn),
                  "propcoco": lambda: R.proposals_coco(anchors_fn, False),
                  "propcoco_train": lambda: R.proposals_coco(anchors_fn, True)}
ROI_CASES = {"roi255": R.roi_pooling_debug255, "roismall7": lambda: R.roi_pooling_small(7),
             "roismall14": lambda: R.roi_pooling_small(14), "roismall1": lambda: R.roi_pooling_small(1)}
TARGET_CASES = {"tgt0": lambda: R.targets_cfg3(0), "tgt1": lambda: R.targets_cfg3(1), "tgt2": lambda: R.targets_cfg3(2),
                "tgttoy": R.targets_toy, "tgtfew": R.targets_few_positives}
DET_CASES = {"det863": R.detection_debug863, "detcoco": R.detection_coco, "dettoy": R.detection_toy_many_per_class}


# ------------------------------------------------------------------------------------------ Proposals
@pytest.mark.parametrize("name", list(PROPOSAL_CASES))
def test_proposals_oracle_equals_reference_run(G, name):
    rec = PROPOSAL_CASES[name]()
    c = rec["conf"]
    n_after = c.POST_NMS_ROIS_TRAINING if rec["training"] else c.POST_NMS_ROIS_INFERENCE
    out, d = oracle.proposal_forward(rec["probs"], rec["bbox"], rec["anchors"], c.RPN_BBOX_STDDEV, c.PRE_NMS_ROIS_COUNT,
                                     n_after, c.RPN_NMS_THRESHOLD, debug=True)
    out = np.where(np.isnan(out), f32(0), out)         # DEBUG=True scrubs NaNs (proposals_tf.py:202-209)
    bits(d["ix"], G[f"{name}/ix"], "ix")
    for k in ("scores", "bbox_delta", "anchors", "anchor_delta", "anchor_delta_clipped"):
        bits(d[k], G[f"{name}/{k}"], k)
    bits(out, G[f"{name}/proposals"], "proposals")


@pytest.mark.parametrize("name", ["prop325", "proptoy"])
def test_proposals_numpy_oracle_equals_reference_run(G, name):
    rec = PROPOSAL_CASES[name]()
    out, d = np_layers.proposals(rec["conf"], rec["probs"], rec["bbox"], rec["anchors"], training=rec["training"])
    out = np.where(np.isnan(out), f32(0), out)
    bits(d["ix"], G[f"{name}/ix"], "ix")
    bits(d["anchor_delta_clipped"], G[f"{name}/anchor_delta_clipped"], "clipped")
    bits(out, G[f"{name}/proposals"], "proposals")


# ------------------------------------------------------------------------------------------ roi_pooling
def derived_roi_debug(roi_level, levels):
    """box_to_level / sorting_tensor / ix of maskrcnn.py:128-173 as functions of roi_level (they are pure index
    plumbing): per level in order, the (batch, box) coordinates of its ROIs row-major, then a running range column;
    key = batch*100000 + box; ix = positions sorted by key ascending (top_k descending, reversed: for equal keys
    the HIGHER position comes first)."""
    b2l = np.concatenate([np.argwhere(roi_level == lv) for lv in levels], axis=0).astype(np.int32)
    b2l = np.concatenate([b2l, np.arange(b2l.shape[0], dtype=np.int32)[:, None]], axis=1)
    key = b2l[:, 0] * 100000 + b2l[:, 1]
    ix = np.argsort(-key.astype(np.int64), kind="stable")[::-1].astype(np.int32)
    return b2l, key, ix


@pytest.mark.parametrize("name", list(ROI_CASES))
def test_roi_pooling_oracle_equals_reference_run(G, name):
    rec = ROI_CASES[name]()
    ph, pw = rec["pool_shape"]
    pooled, lv = oracle.pyramid_roi_align(rec["fmaps"], rec["proposals"], rec["image_shape"][0], rec["image_shape"][1],
                                          ph, pw, min(rec["levels"]))
    bits(lv, G[f"{name}/roi_level"], "roi_level")
    assert list(pooled.shape) == G[f"{name}/pooled_shape"].tolist()
    assert sha(pooled).tolist() == G[f"{name}/pooled_sha256"].tolist(), "pooled_rois differ from the reference run"
    if f"{name}/pooled" in G:
        bits(pooled, G[f"{name}/pooled"], "pooled")
    else:
        bits(pooled[0, ::41, :, :, ::32], G[f"{name}/pooled_sample"], "pooled sample")
    b2l, key, ix = derived_roi_debug(lv, rec["levels"])
    bits(b2l, G[f"{name}/box_to_level"], "box_to_level")
    bits(key, G[f"{name}/sorting_tensor"], "sorting_tensor")
    bits(ix, G[f"{name}/ix"], "ix")


@pytest.mark.parametrize("name", ["roismall7", "roismall1"])
def test_roi_pooling_numpy_oracle_equals_reference_run(G, name):
    rec = ROI_CASES[name]()
    pooled, lv = np_layers.roi_pooling(rec["image_shape"], rec["pool_shape"], rec["levels"], rec["proposals"], rec["fmaps"])
    bits(lv, G[f"{name}/roi_level"], "roi_level")
    bits(pooled, G[f"{name}/pooled"], "pooled")


# ------------------------------------------------------------------------------------------ BuildDetectionTargets
def reference_target_debug(rec, rois, cls, deltas, dbg):
    """The reference's 21-key debug dict (data_processor.py:629-652) assembled from the oracle's outputs + its raw
    debug arrays (iou rows/cols in compacted order, sampled index lists, counts, assignment)."""
    props, gt_cls, gt_box = rec["proposals"], rec["gt_class_ids"], rec["gt_bboxes"]
    n_prop, n_gt, _, _, pos_count, neg_count = (int(v) for v in dbg["counts"])
    nzp = (props != 0).any(axis=1)
    nzg = gt_cls != 0
    sp, sn = dbg["sampled_pos"][:pos_count].astype(np.int64), dbg["sampled_neg"][:neg_count].astype(np.int64)
    iou = dbg["iou"][:n_prop, :n_gt]
    assign = dbg["gt_assignment"][:pos_count].astype(np.int64)
    R = rec["conf"].MRCNN_TRAIN_ROIS_PER_IMAGE
    return dict(non_zero_proposals=nzp, prop_corresponding_gt_non_zero=props[nzp], non_zeros_gt_box=nzg,
                gt_boxes_non_zero=gt_box[nzg], gt_class_ids_non_zero=gt_cls[nzg], iou=iou,
                roi_iou_max=dbg["roi_iou_max"][:n_prop], pos_indices_05more=sp, neg_indices_05more=sn,
                num_pos_inst=np.array(int(R * 0.33)), pos_indices=sp, pos_count=np.array(pos_count, np.int32),
                neg_cnt=np.array(int(f32(1 / 0.33) * f32(pos_count)) - pos_count, np.int32), neg_indices=sn,
                pos_rois=rois[:pos_count], neg_rois=rois[pos_count:pos_count + neg_count], pos_iou=iou[sp],
                roi_gt_box_assignment=assign, roi_gt_class_ids=cls[0, :pos_count],
                roi_gt_boxes=gt_box[nzg][assign], roi_gt_box_deltas=deltas[:pos_count])


def check_target_debug(G, name, d):
    keys = [k.split("/")[-1] for k in G.files if k.startswith(f"{name}/dbg/")]
    assert len(keys) >= 20
    for k in keys:
        if k == "iou_shape":
            assert list(d["iou"].shape) == G[f"{name}/dbg/iou_shape"].tolist()
        elif k == "iou_sha256":
            assert sha(np.ascontiguousarray(d["iou"], f32)).tolist() == G[f"{name}/dbg/iou_sha256"].tolist(), "iou"
        else:
            bits(d[k], G[f"{name}/dbg/{k}"], f"debug[{k}]")


@pytest.mark.parametrize("name", list(TARGET_CASES))
def test_detection_targets_oracle_equals_reference_run(G, name):
    rec = TARGET_CASES[name]()
    c = rec["conf"]
    rois, cls, deltas, dbg = oracle.detection_targets(rec["proposals"], rec["gt_class_ids"], rec["gt_bboxes"],
                                                      rec["perm_pos"], rec["perm_neg"], c.MRCNN_TRAIN_ROIS_PER_IMAGE,
                                                      c.BBOX_STD_DEV)
    bits(rois, G[f"{name}/rois"], "rois")
    bits(cls, G[f"{name}/roi_gt_class_ids"], "roi_gt_class_ids")
    bits(deltas, G[f"{name}/roi_gt_box_deltas"], "roi_gt_box_deltas")
    check_target_debug(G, name, reference_target_debug(rec, rois, cls, deltas, dbg))


@pytest.mark.parametrize("name", ["tgttoy", "tgtfew"])
def test_detection_targets_numpy_oracle_equals_reference_run(G, name):
    rec = TARGET_CASES[name]()
    rois, cls, deltas, _ = np_layers.build_detection_target(rec["conf"], rec["proposals"], rec["gt_class_ids"],
                                                            rec["gt_bboxes"], rec["perm_pos"], rec["perm_neg"])
    bits(rois, G[f"{name}/rois"], "rois")
    bits(cls, G[f"{name}/roi_gt_class_ids"], "cls")
    bits(deltas, G[f"{name}/roi_gt_box_deltas"], "deltas")


# ------------------------------------------------------------------------------------------ DetectionLayer
def reference_detection_debug(rec, d):
    """The 11 items of DetectionLayer.debug_outputs() (detection.py:268-279) from the oracle's intermediates."""
    B, N = d["class_ids"].shape
    mesh = np.repeat(np.arange(B, dtype=np.int32)[:, None], N, axis=1)
    indices = np.tile(np.arange(N, dtype=np.int32), (B, 1))
    ixs = np.stack([mesh, indices, d["class_ids"]], axis=2)
    bbox_delta = (rec["bbox"] * np.asarray(rec["conf"].BBOX_STD_DEV, f32))[mesh, indices, d["class_ids"]]
    keep = d["keep_mask"].astype(bool)
    return dict(class_ids=d["class_ids"], indices=indices, mesh=mesh, ixs=ixs, class_scores=d["class_scores"],
                bbox_delta=bbox_delta, refined_proposals=d["refined_proposals"],
                clipped_proposals_list=[d["clipped_proposals"][b][None] for b in range(B)],
                pre_nms_class_ids_list=[d["class_ids"][b][keep[b]] for b in range(B)],
                pre_nms_scores_list=[d["class_scores"][b][keep[b]] for b in range(B)],
                pre_nms_proposals_list=[d["clipped_proposals"][b][keep[b]] for b in range(B)])


def check_detection_debug(G, name, dd):
    for k, v in dd.items():
        if isinstance(v, list):
            for i, vi in enumerate(v):
                bits(vi, G[f"{name}/dbg/{k}/{i}"], f"{k}[{i}]")
        else:
            bits(v, G[f"{name}/dbg/{k}"], k)


@pytest.mark.parametrize("name", list(DET_CASES))
def test_detection_layer_oracle_equals_reference_run(G, name):
    rec = DET_CASES[name]()
    c = rec["conf"]
    win = oracle.norm_boxes(rec["window"], rec["image_shape"][:2])
    det, d = oracle.detection_forward(rec["proposals"], rec["probs"], rec["bbox"], win, c.BBOX_STD_DEV,
                                      c.DETECTION_MIN_THRESHOLD, c.DETECTION_NMS_THRESHOLD,
                                      c.DETECTION_POST_NMS_INSTANCES, debug=True)
    bits(det, G[f"{name}/detections"], "detections")
    check_detection_debug(G, name, reference_detection_debug(rec, d))


@pytest.mark.parametrize("name", ["det863", "dettoy"])
def test_detection_layer_numpy_oracle_equals_reference_run(G, name):
    rec = DET_CASES[name]()
    win = oracle.norm_boxes(rec["window"], rec["image_shape"][:2])
    det = np_layers.detection_layer(rec["conf"], win, rec["proposals"], rec["probs"], rec["bbox"])
    bits(det, G[f"{name}/detections"], "detections")


def test_unmold_oracle_equals_reference_run(G):
    rec = R.detection_coco()
    for b in range(2):
        boxes, cids, scores = oracle.unmold_detection([720, 1280, 3], [1024, 1024, 3], G["detcoco/detections"][b], rec["window"][b])
        bits(boxes, G[f"detcoco/unmold/{b}/boxes"], "boxes")
        bits(cids, G[f"detcoco/unmold/{b}/class_ids"], "class_ids")
        bits(scores, G[f"detcoco/unmold/{b}/scores"], "scores")


# ------------------------------------------------------------------------------------------ norm_boxes_tf
def test_norm_boxes_tf_oracle_equals_reference_run(G):
    rec = R.norm_boxes_tf_case()
    for i, shp in enumerate(rec["shapes"]):
        bits(oracle.norm_boxes_tf(rec["boxes"][i], shp), G[f"normtf/{i}"], f"norm_boxes_tf {shp}")


# ------------------------------------------------------------------------------------------ the shim itself
def test_tf_shim_dtype_rules():
    import tf_shim
    tf = tf_shim.install()
    x = tf.constant(np.array([1.5, 2.5, -0.5], f32))
    assert (x * np.array([0.1, 0.1, 0.2])).a.dtype == f32                        # numpy operand -> tensor dtype
    assert ((1 / 0.33) * tf.cast(tf.constant(3), tf.float32)).a == f32(f32(1 / 0.33) * f32(3))
    assert tf.round(x).a.tolist() == [2.0, 2.0, -0.0]                            # half to even
    assert tf.cast(tf.constant(np.array([np.nan, -np.inf, 3.9], f32)), tf.int32).a.tolist() == [-2 ** 31, -2 ** 31, 3]
    with pytest.raises(TypeError):
        x + tf.constant(np.array([1, 2, 3], np.int32))                           # mixed dtypes raise like TensorFlow
    w = tf.where(tf.constant(np.array([[0, 1], [1, 1]])) > 0)
    assert w.a.dtype == np.int64 and w.a.tolist() == [[0, 1], [1, 0], [1, 1]]
    u = tf.unique(tf.constant(np.array([5, 3, 5, 7, 3], np.int32)))
    assert u.y.a.tolist() == [5, 3, 7] and u.idx.a.tolist() == [0, 1, 0, 2, 1]
    s = tf.sparse_tensor_to_dense(tf.sets.set_intersection(tf.constant(np.array([[9, 2, 4, 4]], np.int64)),
                                                           tf.constant(np.array([[4, 9, 1]], np.int64))))
    assert s.a.tolist() == [[4, 9]]
    tf_shim.set_shuffle_perms([np.array([3, 0, 5, 2, 1, 4])])
    assert tf.random_shuffle(tf.constant(np.array([10, 11, 12, 13], np.int64))).a.tolist() == [13, 10, 12, 11]
    assert tf.nn.top_k(tf.constant(np.array([[1., 3., 3., 2.]], f32)), 3).indices.a.tolist() == [[1, 2, 3]]
