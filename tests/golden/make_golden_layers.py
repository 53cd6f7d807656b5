"""Regenerates tests/golden/reference_layers.npz by RUNNING THE REFERENCE'S OWN LAYER CLASSES, unmodified, from
/root/reference — `Proposals` (proposals_tf.py), `MaskRCNN.roi_pooling` (maskrcnn.py), `BuildDetectionTargets`
(data_processor.py), `DetectionLayer` (detection.py) and `utils.norm_boxes_tf` — through the numpy-eager TensorFlow
stand-in tests/tf_shim (see its docstring for exactly what is emulated and what delegates to the oracle's restatement
of the three TF C++ kernels).  Every `DEBUG=True` intermediate the classes expose is frozen next to the outputs.

Build container only (needs /root/reference):   python tests/golden/make_golden_layers.py
The inputs come from tests/golden/layer_recipes.py (seeded; the tests regenerate them), so the .npz holds outputs
only: full arrays where they are small, sha256 digests + strided samples where they are not, and every member above
golden_sample.MAX_WHOLE elements as its shape, digest and a seeded row sample (golden_sample.shrink).
"""
import hashlib
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = "/root/reference"
OUT = os.path.join(HERE, "reference_layers.npz")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

import golden_sample  # noqa: E402
import layer_recipes as R  # noqa: E402
import tf_shim  # noqa: E402

from make_golden_layers_keys import DET_DEBUG_KEYS  # noqa: E402


def digest(a):
    a = np.ascontiguousarray(a)
    return np.frombuffer(hashlib.sha256(a.tobytes()).digest(), np.uint8)


def import_reference():
    tf = tf_shim.install()
    sys.path.insert(0, REF)
    cwd = os.getcwd()
    os.chdir(tempfile.mkdtemp())          # the reference truncates ./logfile.log at import
    try:
        from MaskRCNN.building_blocks import data_processor, detection, maskrcnn, proposals_tf, utils
        from MaskRCNN.config import config as ref_config
    finally:
        os.chdir(cwd)
    return tf, proposals_tf, maskrcnn, data_processor, detection, utils, ref_config


def ref_conf(ref_config, recipe_conf):
    """The reference's own config class, with the recipe's overrides applied as a subclass (shapes.py style)."""
    over = {}
    for k in dir(R.RefConfig):
        if k.startswith("_"):
            continue
        want, have = getattr(recipe_conf, k), getattr(ref_config, k)
        if isinstance(have, np.ndarray) or isinstance(want, np.ndarray):
            same = np.array_equal(np.asarray(want), np.asarray(have))
        else:
            same = list(np.atleast_1d(want)) == list(np.atleast_1d(have))
        if not same:
            over[k] = want
    if recipe_conf is R.RefConfig:
        assert not over, f"layer_recipes.RefConfig drifted from MaskRCNN/config.py: {over}"
    return type("conf", (ref_config,), over)


def main():
    tf, proposals_tf, maskrcnn, data_processor, detection, utils, ref_config = import_reference()
    sess = tf.Session()
    g = {}

    def anchors_fn(conf, batch):
        shapes = utils.get_resnet_stage_shapes(conf, conf.IMAGE_SHAPE)
        return utils.gen_anchors(conf.IMAGE_SHAPE, batch, conf.RPN_ANCHOR_SCALES, conf.RPN_ANCHOR_RATIOS, shapes,
                                 conf.RESNET_STRIDES, conf.RPN_ANCHOR_STRIDE)

    # ------------------------------------------------------------------ Proposals (proposals_tf.py:98-326)
    for name, rec in (("prop325", R.proposals_debug325()), ("proptoy", R.proposals_toy(anchors_fn)),
                      ("propcoco", R.proposals_coco(anchors_fn, False)), ("propcoco_train", R.proposals_coco(anchors_fn, True))):
        obj = proposals_tf.Proposals(ref_conf(ref_config, rec["conf"]), rec["batch"], tf.constant(rec["probs"]),
                                     tf.constant(rec["bbox"]), tf.constant(rec["anchors"]), training=rec["training"], DEBUG=True)
        bbox_delta, ix, scores, anchors, anchor_delta = sess.run(list(obj.debug_outputs()))
        clipped = sess.run(obj.get_anchors_delta_clipped())
        proposals = sess.run(obj.get_proposals())
        assert proposals.dtype == np.float32 and ix.dtype == np.int32
        g[f"{name}/proposals"], g[f"{name}/ix"] = proposals, ix
        g[f"{name}/scores"], g[f"{name}/bbox_delta"], g[f"{name}/anchors"] = scores, bbox_delta, anchors
        g[f"{name}/anchor_delta"], g[f"{name}/anchor_delta_clipped"] = anchor_delta, clipped
        print(name, proposals.shape, "kept", [(np.abs(p).sum(1) != 0).sum() for p in proposals])

    # ------------------------------------------------------------------ MaskRCNN.roi_pooling (maskrcnn.py:74-187)
    for name, rec in (("roi255", R.roi_pooling_debug255()), ("roismall7", R.roi_pooling_small(7)),
                      ("roismall14", R.roi_pooling_small(14)), ("roismall1", R.roi_pooling_small(1))):
        obj = maskrcnn.MaskRCNN(image_shape=rec["image_shape"], pool_shape=rec["pool_shape"], num_classes=4,
                                levels=rec["levels"], proposals=rec["proposals"], feature_maps=rec["fmaps"],
                                type="keras", DEBUG=True)
        roi_level, box_to_level, sorting_tensor, ix = sess.run(list(obj.debug_outputs()[:4]))
        pooled = sess.run(obj.get_pooled_rois())
        assert pooled.dtype == np.float32 and pooled.shape[0] == 1
        g[f"{name}/roi_level"], g[f"{name}/box_to_level"] = roi_level, box_to_level
        g[f"{name}/sorting_tensor"], g[f"{name}/ix"] = sorting_tensor, ix
        g[f"{name}/pooled_shape"] = np.array(pooled.shape)
        g[f"{name}/pooled_sha256"] = digest(pooled)
        if pooled.nbytes <= 2 << 20:
            g[f"{name}/pooled"] = pooled
        else:
            g[f"{name}/pooled_sample_rows"] = np.arange(0, pooled.shape[1], 41)
            g[f"{name}/pooled_sample"] = pooled[0, ::41, :, :, ::32].copy()
        print(name, pooled.shape, "levels", np.bincount(roi_level.ravel(), minlength=6)[2:])
        del obj, pooled

    # ------------------------------------------------------------------ BuildDetectionTargets (data_processor.py:430-658)
    for name, rec in (("tgt0", R.targets_cfg3(0)), ("tgt1", R.targets_cfg3(1)), ("tgt2", R.targets_cfg3(2)),
                      ("tgttoy", R.targets_toy()), ("tgtfew", R.targets_few_positives())):
        tf_shim.set_shuffle_perms([rec["perm_pos"], rec["perm_neg"]])
        obj = data_processor.BuildDetectionTargets(ref_conf(ref_config, rec["conf"]), tf.constant(rec["proposals"]),
                                                   tf.constant(rec["gt_class_ids"]), tf.constant(rec["gt_bboxes"]), DEBUG=True)
        rois, cls, deltas = sess.run(list(obj.get_target_rois()))
        dbg = sess.run(obj.debug_outputs())
        g[f"{name}/rois"], g[f"{name}/roi_gt_class_ids"], g[f"{name}/roi_gt_box_deltas"] = rois, cls, deltas
        for k, v in dbg.items():
            v = np.asarray(v)
            if k == "iou" and v.nbytes > 1 << 18:
                g[f"{name}/dbg/iou_sha256"] = digest(v)
                g[f"{name}/dbg/iou_shape"] = np.array(v.shape)
                continue
            g[f"{name}/dbg/{k}"] = v
        print(name, "pos", int(dbg["pos_count"]), "neg", int(np.asarray(dbg["neg_indices"]).shape[0]), "keys", len(dbg))

    # ------------------------------------------------------------------ DetectionLayer (detection.py:56-279)
    for name, rec in (("det863", R.detection_debug863()), ("detcoco", R.detection_coco()),
                      ("dettoy", R.detection_toy_many_per_class())):
        obj = detection.DetectionLayer(ref_conf(ref_config, rec["conf"]), rec["image_shape"], rec["proposals"].shape[0],
                                       rec["window"], rec["proposals"], rec["probs"], rec["bbox"], DEBUG=True)
        det = sess.run(obj.get_detections())
        dbg = sess.run(list(obj.debug_outputs()))
        assert det.dtype == np.float32
        g[f"{name}/detections"] = det
        for k, v in zip(DET_DEBUG_KEYS, dbg):
            if isinstance(v, list):
                for i, vi in enumerate(v):
                    g[f"{name}/dbg/{k}/{i}"] = np.asarray(vi)
            else:
                g[f"{name}/dbg/{k}"] = np.asarray(v)
        print(name, det.shape, "detections/img", [(d[:, 4] > 0).sum() for d in det])

    # unmold_detection on the COCO-shape detections (detection.py:8-53; numpy, host)
    import contextlib
    import io
    rec = R.detection_coco()
    with contextlib.redirect_stdout(io.StringIO()):
        for b in range(2):
            boxes, cids, scores = detection.unmold_detection([720, 1280, 3], [1024, 1024, 3], g["detcoco/detections"][b], rec["window"][b])
            g[f"detcoco/unmold/{b}/boxes"], g[f"detcoco/unmold/{b}/class_ids"], g[f"detcoco/unmold/{b}/scores"] = boxes, cids, scores

    # ------------------------------------------------------------------ utils.norm_boxes_tf (utils.py:198-210)
    rec = R.norm_boxes_tf_case()
    for i, shp in enumerate(rec["shapes"]):
        out = sess.run(utils.norm_boxes_tf(tf.constant(rec["boxes"][i]), shp))
        assert out.dtype == np.float32
        g[f"normtf/{i}"] = out
    # SURVEY §4 G4: the notebook's recorded normalised toy GT boxes
    want = np.array([[0.04724409, 0.57480317, 0.42519686, 0.96850395], [0.40944883, 0.36220473, 0.88188976, 0.83464569],
                     [0.44881889, 0.23622048, 0.76377952, 0.55118108]])
    assert np.allclose(g["normtf/0"][:3], want, rtol=0, atol=1e-7), g["normtf/0"][:3]

    np.savez_compressed(OUT, **golden_sample.shrink(g))
    print(f"wrote {OUT}: {len(g)} arrays, {os.path.getsize(OUT) / 1e6:.2f} MB")


if __name__ == "__main__":
    main()
