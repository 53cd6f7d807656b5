"""GPU parity against goldens produced by the REFERENCE'S OWN layer classes (tests/golden/reference_layers.npz, written
by tests/golden/make_golden_layers.py: proposals_tf.py / maskrcnn.py / data_processor.py / detection.py / utils.py run
unmodified through tests/tf_shim). The CUDA path is driven through the reference-named classes with DEBUG=True, read
back the way the reference's own debug() functions do, and every output and every DEBUG intermediate must equal the
frozen reference run bit for bit. Nothing here calls the oracle: the expected values are the files.
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
from test_reference_layer_goldens import (DET_CASES, PROPOSAL_CASES, ROI_CASES, TARGET_CASES, bits, sha)  # noqa: E402

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu
f32 = np.float32


@pytest.fixture(scope="module", autouse=True)
def _need_cuda():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (there is no CPU path)")


@pytest.fixture(scope="module")
def G():
    return golden_sample.Golden(os.path.join(HERE, "golden", "reference_layers.npz"))


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    if isinstance(t, (list, tuple)):
        return [host(v) for v in t]
    if isinstance(t, torch.Tensor):
        torch.cuda.synchronize()
        return t.detach().cpu().numpy()
    return np.asarray(t)


class _AnchorsOnDevice:
    """The recipes take an anchors_fn(conf, batch) -> numpy; here it is the package's own GPU anchor generator."""

    def __call__(self, conf, batch):
        from objectdetection_b200 import utils
        shapes = utils.get_resnet_stage_shapes(conf, conf.IMAGE_SHAPE)
        return host(utils.gen_anchors(conf.IMAGE_SHAPE, batch, conf.RPN_ANCHOR_SCALES, conf.RPN_ANCHOR_RATIOS, shapes,
                                      conf.RESNET_STRIDES, conf.RPN_ANCHOR_STRIDE))


def _proposal_case(name):
    fn = _AnchorsOnDevice()
    return {"prop325": R.proposals_debug325, "proptoy": lambda: R.proposals_toy(fn),
            "propcoco": lambda: R.proposals_coco(fn, False), "propcoco_train": lambda: R.proposals_coco(fn, True)}[name]()


@pytest.mark.parametrize("name", list(PROPOSAL_CASES))
def test_proposals_equal_reference_run(G, name):
    from objectdetection_b200 import Proposals
    rec = _proposal_case(name)
    obj = Proposals(rec["conf"], rec["batch"], cu(rec["probs"]), cu(rec["bbox"]), cu(rec["anchors"]),
                    training=rec["training"], DEBUG=True)
    bbox_delta, ix, scores, anchors, anchor_delta = host(obj.debug_outputs())
    bits(ix, G[f"{name}/ix"], "ix")
    bits(scores, G[f"{name}/scores"], "scores")
    bits(bbox_delta, G[f"{name}/bbox_delta"], "bbox_delta")
    bits(anchors, G[f"{name}/anchors"], "anchors")
    bits(anchor_delta, G[f"{name}/anchor_delta"], "anchor_delta")
    bits(host(obj.get_anchors_delta_clipped()), G[f"{name}/anchor_delta_clipped"], "anchor_delta_clipped")
    bits(host(obj.get_proposals()), G[f"{name}/proposals"], "proposals")
    g = obj.get_proposal_graph()
    assert set(g) == {"rpn_class_probs", "rpn_bbox", "input_anchors", "proposals"}


@pytest.mark.parametrize("name", list(ROI_CASES))
def test_roi_pooling_equals_reference_run(G, name):
    from objectdetection_b200 import MaskRCNN
    rec = ROI_CASES[name]()
    obj = MaskRCNN(image_shape=rec["image_shape"], pool_shape=rec["pool_shape"], num_classes=4, levels=rec["levels"],
                   proposals=cu(rec["proposals"]), feature_maps=[cu(f) for f in rec["fmaps"]], type="keras", DEBUG=True)
    roi_level, box_to_level, sorting_tensor, ix = host(list(obj.debug_outputs()[:4]))
    pooled = host(obj.get_pooled_rois())
    bits(roi_level, G[f"{name}/roi_level"], "roi_level")
    bits(box_to_level, G[f"{name}/box_to_level"], "box_to_level")
    bits(sorting_tensor, G[f"{name}/sorting_tensor"], "sorting_tensor")
    bits(ix, G[f"{name}/ix"], "ix")
    assert list(pooled.shape) == G[f"{name}/pooled_shape"].tolist()
    if f"{name}/pooled" in G:
        bits(pooled, G[f"{name}/pooled"], "pooled_rois")
    else:
        bits(pooled[0, ::41, :, :, ::32], G[f"{name}/pooled_sample"], "pooled_rois sample")
    assert sha(pooled).tolist() == G[f"{name}/pooled_sha256"].tolist(), "pooled_rois differ from the reference run"


@pytest.mark.parametrize("name", list(TARGET_CASES))
def test_detection_targets_equal_reference_run(G, name):
    from objectdetection_b200 import BuildDetectionTargets
    rec = TARGET_CASES[name]()
    obj = BuildDetectionTargets(rec["conf"], cu(rec["proposals"]), cu(rec["gt_class_ids"]), cu(rec["gt_bboxes"]),
                                DEBUG=True, perm_pos=cu(rec["perm_pos"]), perm_neg=cu(rec["perm_neg"]))
    rois, cls, deltas = host(list(obj.get_target_rois()))
    bits(rois, G[f"{name}/rois"], "rois")
    bits(cls, G[f"{name}/roi_gt_class_ids"], "roi_gt_class_ids")
    bits(deltas, G[f"{name}/roi_gt_box_deltas"], "roi_gt_box_deltas")
    d = obj.debug_outputs()
    keys = sorted({k.split("/")[2] for k in G.files if k.startswith(f"{name}/dbg/")} - {"iou_shape", "iou_sha256"})
    want_keys = set(keys) | ({"iou"} if f"{name}/dbg/iou_sha256" in G else set())
    assert set(d) == want_keys and len(d) == 21, sorted(set(d) ^ want_keys)
    for k in keys:
        bits(host(d[k]), G[f"{name}/dbg/{k}"], f"debug[{k}]")
    if f"{name}/dbg/iou_sha256" in G:
        iou = np.ascontiguousarray(host(d["iou"]), f32)
        assert list(iou.shape) == G[f"{name}/dbg/iou_shape"].tolist()
        assert sha(iou).tolist() == G[f"{name}/dbg/iou_sha256"].tolist(), "iou differs from the reference run"


@pytest.mark.parametrize("name", list(DET_CASES))
@pytest.mark.parametrize("window_on_device", [False, True])
def test_detection_layer_equals_reference_run(G, name, window_on_device):
    from objectdetection_b200 import DetectionLayer
    from test_reference_layer_goldens import check_detection_debug
    from make_golden_layers_keys import DET_DEBUG_KEYS
    rec = DET_CASES[name]()
    window = cu(rec["window"]) if window_on_device else rec["window"]
    obj = DetectionLayer(rec["conf"], rec["image_shape"], rec["proposals"].shape[0], window, cu(rec["proposals"]),
                         cu(rec["probs"]), cu(rec["bbox"]), DEBUG=True)
    bits(host(obj.get_detections()), G[f"{name}/detections"], "detections")
    dbg = obj.debug_outputs()
    assert len(dbg) == len(DET_DEBUG_KEYS)
    check_detection_debug(G, name, {k: host(v) for k, v in zip(DET_DEBUG_KEYS, dbg)})


def test_unmold_equals_reference_run(G):
    from objectdetection_b200.detection import unmold_detection
    rec = R.detection_coco()
    for b in range(2):
        boxes, cids, scores = unmold_detection([720, 1280, 3], [1024, 1024, 3], G["detcoco/detections"][b], rec["window"][b])
        assert boxes.dtype == np.int32 and cids.dtype == np.int32
        bits(boxes, G[f"detcoco/unmold/{b}/boxes"], "boxes")
        bits(cids, G[f"detcoco/unmold/{b}/class_ids"], "class_ids")
        bits(scores, G[f"detcoco/unmold/{b}/scores"], "scores")


def test_norm_boxes_tf_equals_reference_run(G):
    from objectdetection_b200 import utils
    rec = R.norm_boxes_tf_case()
    for i, shp in enumerate(rec["shapes"]):
        bits(host(utils.norm_boxes_tf(cu(rec["boxes"][i]), shp)), G[f"normtf/{i}"], f"norm_boxes_tf {shp}")


def test_norm_boxes_device_equals_numpy_formula(golden):
    """utils.norm_boxes on a CUDA tensor (int32 / float32 / float64 pixels) == the reference's numpy formula."""
    from objectdetection_b200 import utils
    rs = np.random.RandomState(3)
    for dt in (np.int32, np.float32, np.float64):
        px = (rs.random_sample((40, 4)) * 1024).astype(dt)
        for shp in ((1024, 1024), (600, 1000), (128, 128)):
            bits(host(utils.norm_boxes(cu(px), shp)), utils.norm_boxes(px, shp), f"norm_boxes {dt} {shp}")
    got = host(utils.norm_boxes(cu(np.asarray(golden["norm_in_window"]).reshape(-1, 4)), (1024, 1024)))
    bits(got, np.asarray(golden["norm_out_window"]).reshape(-1, 4), "G5 window (reference-run golden)")
