"""GPU parity: the CUDA path (through the reference-named layer classes -> C ABI -> sm_100a kernels) against the CPU
oracle on identical seeded inputs. Integer / index outputs must be bit-exact; decoded boxes and deltas are asserted
bit-exact as well (the oracle and the kernels share the numeric contract) with the north-star tolerance (rtol 1e-5)
as the documented fallback bound; ROIAlign features rtol 1e-4."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import _synth  # noqa: E402

import oracle  # noqa: E402
from objectdetection_b200.config import ShapesConfig, config as Conf  # noqa: E402

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu
f32 = np.float32
STRIDES = [4, 8, 16, 32, 64]


@pytest.fixture(scope="module", autouse=True)
def _need_cuda():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (there is no CPU path)")


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    torch.cuda.synchronize()
    return t.detach().cpu().numpy()


def assert_bits(a, b, what=""):
    a, b = np.asarray(a, f32), np.asarray(b, f32)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    same = (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))
    if not same.all():
        bad = np.argwhere(~same)
        raise AssertionError(f"{what}: {bad.shape[0]} of {a.size} differ; first {bad[:3].tolist()} "
                             f"got {a[tuple(bad[0])]!r} want {b[tuple(bad[0])]!r}; "
                             f"max rel {np.nanmax(np.abs(a - b) / (np.abs(b) + 1e-30)):.3e}")


# ------------------------------------------------------------------ anchors
def test_gen_anchors_bit_exact():
    from objectdetection_b200 import utils
    for shape, scales, ratios, astride in (([128, 128, 3], (8, 16, 32, 64, 128), [0.5, 1, 2], 1),
                                           ([1024, 1024, 3], (32, 64, 128, 256, 512), [0.5, 1, 2], 1),
                                           ([192, 320, 3], (16, 32, 64, 128, 256), [0.5, 1, 2, 3], 2)):
        c = Conf()
        shapes = utils.get_resnet_stage_shapes(c, shape)
        got = host(utils.gen_anchors(shape, 2, scales, ratios, shapes, STRIDES, astride))
        want = oracle.gen_anchors(shape, 2, scales, ratios, shapes, STRIDES, astride)
        assert_bits(got, want, f"anchors {shape}")
        gp = host(utils.gen_anchors_pixel_coord(scales, ratios, shapes, STRIDES, astride))
        assert np.array_equal(gp, oracle.gen_anchors_pixel_coord(scales, ratios, shapes, STRIDES, astride))


def test_anchors_golden_on_gpu(golden):
    from objectdetection_b200 import utils
    got = host(utils.gen_anchors([1024, 1024, 3], 1, (32, 64, 128, 256, 512), [0.5, 1, 2], golden["stage_shapes_1024"], STRIDES, 1))
    assert got.shape == (1, 261888, 4)
    assert np.array_equal(got[0, golden["anchors_1024_sample_rows"]], golden["anchors_1024_sample"])
    toy = host(utils.gen_anchors_pixel_coord((8, 16, 32, 64, 128), [0.5, 1, 2], golden["stage_shapes_128"], STRIDES, 1))
    assert np.array_equal(toy, golden["anchors_toy_pixel"])


# ------------------------------------------------------------------ top-k
@pytest.mark.parametrize("rows,cols,k", [(3, 500, 200), (2, 300, 300), (2, 4092, 4092), (2, 261888, 6000), (1, 70000, 20000),
                                         (5, 33, 1)])
def test_topk(rows, cols, k):
    from objectdetection_b200.proposals import top_k
    rs = np.random.RandomState(rows * 7 + cols)
    probs = rs.random_sample((rows, cols, 2)).astype(f32)
    if cols <= 4092:
        probs = (np.round(probs * 64) / 64).astype(f32)           # heavy ties
        probs[0, 7 % cols, 1], probs[0, 9 % cols, 1] = -0.0, 0.0
    view = cu(probs)[:, :, 1]                                      # strided view, like proposals_tf.py:153
    v, i = top_k(view, k)
    wv, wi = oracle.topk(probs[:, :, 1], k)
    assert np.array_equal(host(i), wi)
    assert_bits(host(v), wv, "values")


def test_topk_all_equal_scores():
    from objectdetection_b200.proposals import top_k
    s = np.full((2, 10000), 0.5, f32)
    v, i = top_k(cu(s), 777)
    assert np.array_equal(host(i), np.tile(np.arange(777, dtype=np.int32), (2, 1)))


def test_topk_candidate_overflow_and_clustered_scores():
    """The split/tail select keeps the keys of the threshold bucket in a bounded candidate buffer; clustered or tied
    scores overflow it and the tail falls back to the original row. Both must stay exact (ties -> lower index)."""
    from objectdetection_b200.proposals import top_k
    s = np.full((2, 100000), 0.5, f32)                      # one bucket holds everything: 100000 > capacity
    s[1, ::3] = 0.75
    v, i = top_k(cu(s), 1000)
    wv, wi = oracle.topk(s, 1000)
    assert np.array_equal(host(i), wi) and np.array_equal(host(v), wv)
    rs = np.random.RandomState(8)
    c = (0.9 + 0.0001 * rs.random_sample((3, 200000))).astype(f32)   # same exponent + top mantissa bits: one big bucket
    v, i = top_k(cu(c), 6000)
    wv, wi = oracle.topk(c, 6000)
    assert np.array_equal(host(i), wi) and np.array_equal(host(v), wv)


# ------------------------------------------------------------------ decode / clip
def test_apply_box_deltas_and_clip():
    from objectdetection_b200.proposals import apply_box_deltas, clip_boxes_to_01
    rs = np.random.RandomState(1)
    a = rs.random_sample((2, 1031, 4)).astype(f32)
    d = rs.normal(0, 1, size=(2, 1031, 4)).astype(f32)
    dec = host(apply_box_deltas(cu(a), cu(d)))
    want = oracle.apply_box_deltas(a, d)
    assert_bits(dec, want, "apply_box_deltas")
    assert np.allclose(dec, want, rtol=1e-5)
    assert_bits(host(clip_boxes_to_01(cu(want), cu(np.array([0, 0, 1, 1], f32)))), oracle.clip_boxes(want, np.array([0, 0, 1, 1], f32)), "clip")
    win = np.array([[0.1, 0.2, 0.8, 0.9], [0, 0.3, 1, 0.7]], f32)
    assert_bits(host(clip_boxes_to_01(cu(want), cu(win))), oracle.clip_boxes(want, win), "clip per image")


# ------------------------------------------------------------------ NMS
@pytest.mark.parametrize("n,thr", [(300, 0.3), (1000, 0.5), (6000, 0.7), (65, 0.1), (1, 0.5)])
def test_nms(n, thr):
    from objectdetection_b200.proposals import non_max_suppression
    rs = np.random.RandomState(n)
    boxes = np.stack([_synth.random_boxes(rs, n, flip=True) for _ in range(2)])
    if n > 10:
        boxes[0, 5] = boxes[0, 6]
        boxes[0, 10, 2:] = boxes[0, 10, :2]
    scores = (rs.randint(0, 200, (2, n)) / 200).astype(f32)
    for max_out in sorted({1, min(100, n), n}):
        keep, num = non_max_suppression(cu(boxes), cu(scores), max_out, thr)
        keep, num = host(keep), host(num)
        for b in range(2):
            want = oracle.nms(boxes[b], scores[b], max_out, thr)
            assert num[b] == want.shape[0], (b, max_out)
            assert np.array_equal(keep[b, :num[b]], want) and np.all(keep[b, num[b]:] == -1)


@pytest.mark.parametrize("K,max_out", [(6000, 1000), (12000, 2000), (20000, 500), (6000, 40), (8000, 8000), (3000, 3000), (200, 200)])
def test_nms_two_rounds_on_clustered_boxes(K, max_out):
    """max_out << K runs the NMS in two rounds (rows of the first 1.5 x max_out boxes, then - decided on the device -
    the rest, with the scan state carried over). Heavily clustered boxes force the second round; ragged num_valid;
    K = 20000 takes the unstaged (global-memory) scan; max_out = K is a single round with 3 (K = 8000), 8 (K = 3000) or
    more ring slots than chunks (K = 200)."""
    from objectdetection_b200.proposals import non_max_suppression
    rs = np.random.RandomState(K + max_out)
    B = 2
    centers = rs.uniform(0.1, 0.9, (B, 60, 2))
    sizes = rs.uniform(0.03, 0.2, (B, 60, 2))
    which = rs.randint(0, 60, (B, K))
    c = np.take_along_axis(centers, which[..., None].repeat(2, -1), 1) + rs.normal(0, 0.004, (B, K, 2))
    hw = np.take_along_axis(sizes, which[..., None].repeat(2, -1), 1) * np.exp(rs.normal(0, 0.06, (B, K, 2)))
    boxes = np.concatenate([c - hw / 2, c + hw / 2], -1).astype(f32)
    scores = rs.random_sample((B, K)).astype(f32)
    nv = np.array([K, K - min(1234, K // 3)], np.int32)
    keep, num = non_max_suppression(cu(boxes), cu(scores), max_out, 0.7, num_valid=nv)
    keep, num = host(keep), host(num)
    visited_all = False
    for b in range(B):
        want = oracle.nms(boxes[b, :nv[b]], scores[b, :nv[b]], max_out, 0.7)
        assert num[b] == want.shape[0], (b, num[b], want.shape[0])
        assert np.array_equal(keep[b, :num[b]], want) and np.all(keep[b, num[b]:] == -1)
        visited_all |= want.shape[0] < max_out
    assert visited_all or max_out == 40      # the clusters are dense enough that the second round had to run


def test_nms_num_valid_and_single_image_form():
    from objectdetection_b200.proposals import non_max_suppression
    rs = np.random.RandomState(4)
    boxes, scores = _synth.random_boxes(rs, 500), rs.random_sample(500).astype(f32)
    k = non_max_suppression(cu(boxes), cu(scores), 500, 0.4)
    assert np.array_equal(host(k), oracle.nms(boxes, scores, 500, 0.4))
    keep, num = non_max_suppression(cu(boxes[None]), cu(scores[None]), 500, 0.4, num_valid=np.array([123], np.int32))
    want = oracle.nms(boxes[:123], scores[:123], 500, 0.4)
    assert host(num)[0] == want.shape[0] and np.array_equal(host(keep)[0, :want.shape[0]], want)


@pytest.mark.parametrize("B,K,max_out,clustered", [(2, 20000, 20000, True), (1, 30000, 21000, False), (3, 13000, 13000, False)])
def test_nms_wide_scan(B, K, max_out, clustered):
    """K beyond the shared-memory ring with max_out ~ K: the multi-CTA scan (bitmap slices, published keep words).
    Clustered boxes (few survivors, all chunks visited), sparse boxes (max_out reached on the way), ragged num_valid."""
    from objectdetection_b200.proposals import non_max_suppression
    rs = np.random.RandomState(K + B)
    if clustered:
        centers, sizes = rs.uniform(0.1, 0.9, (B, 300, 2)), rs.uniform(0.02, 0.1, (B, 300, 2))
        which = rs.randint(0, 300, (B, K))
        c = np.take_along_axis(centers, which[..., None].repeat(2, -1), 1) + rs.normal(0, 0.004, (B, K, 2))
        hw = np.take_along_axis(sizes, which[..., None].repeat(2, -1), 1) * np.exp(rs.normal(0, 0.06, (B, K, 2)))
        boxes = np.concatenate([c - hw / 2, c + hw / 2], -1).astype(f32)
    else:
        boxes = np.stack([_synth.rois_log_uniform(rs, 1, K, image=4096, lo=4, hi=48)[0] for _ in range(B)])
    scores = rs.random_sample((B, K)).astype(f32)
    nv = np.array([K, K - 1777, 64][:B], np.int32)
    keep, num = non_max_suppression(cu(boxes), cu(scores), max_out, 0.5, num_valid=nv)
    keep, num = host(keep), host(num)
    capped = False
    for b in range(B):
        want = oracle.nms(boxes[b, :nv[b]], scores[b, :nv[b]], max_out, 0.5)
        assert num[b] == want.shape[0], (b, num[b], want.shape[0])
        assert np.array_equal(keep[b, :num[b]], want) and np.all(keep[b, num[b]:] == -1)
        capped |= want.shape[0] == max_out
    assert capped == (K == 30000)


def test_nms_stress_100k_boxes():
    """BASELINE config 5: 100,000 boxes, one image, thr 0.5; sqrt(area) log-uniform [8,256] px in 4096^2."""
    from objectdetection_b200.proposals import non_max_suppression
    rs = np.random.RandomState(5)
    boxes = _synth.rois_log_uniform(rs, 1, 100000, image=4096, lo=8, hi=256)[0]
    scores = rs.random_sample(100000).astype(f32)
    keep = host(non_max_suppression(cu(boxes), cu(scores), 100000, 0.5))
    want = oracle.nms(boxes, scores, 100000, 0.5)
    assert np.array_equal(keep, want)
    # idempotence: NMS of the survivors keeps all of them, in the same order
    again = host(non_max_suppression(cu(boxes[keep]), cu(scores[keep]), keep.shape[0], 0.5))
    assert np.array_equal(again, np.arange(keep.shape[0]))


# ------------------------------------------------------------------ ProposalLayer
def _check_proposals(P, probs, bbox, anchors, conf, training=False):
    N = conf.POST_NMS_ROIS_TRAINING if training else conf.POST_NMS_ROIS_INFERENCE
    want, dbg = oracle.proposal_forward(probs, bbox, anchors, conf.RPN_BBOX_STDDEV, conf.PRE_NMS_ROIS_COUNT, N,
                                        conf.RPN_NMS_THRESHOLD, debug=True)
    bbox_delta, ix, scores, anc, anchor_delta = P.debug_outputs()
    assert np.array_equal(host(ix), dbg["ix"])
    assert_bits(host(scores), dbg["scores"], "scores")
    assert_bits(host(bbox_delta), dbg["bbox_delta"], "bbox_delta")
    assert_bits(host(anc), dbg["anchors"], "anchors")
    assert_bits(host(anchor_delta), dbg["anchor_delta"], "anchor_delta")
    assert np.allclose(host(anchor_delta), dbg["anchor_delta"], rtol=1e-5, equal_nan=True)
    assert_bits(host(P.get_anchors_delta_clipped()), dbg["anchor_delta_clipped"], "clipped")
    assert np.array_equal(host(P.num_kept), dbg["num_kept"])
    assert np.array_equal(host(P.keep_idx), dbg["keep_idx"])
    # the DEBUG layer zeroes NaN rows like the reference does in DEBUG mode (proposals_tf.py:202-209)
    assert_bits(host(P.get_proposals()), np.where(np.isnan(want), f32(0), want), "proposals")
    return want


def test_proposals_debug_recipe():
    """proposals_tf.py:331-345: seed 325, (1,4092,{2,4,4}) uniform inputs, COCO config."""
    from objectdetection_b200 import Proposals
    np.random.seed(325)
    probs = np.array(np.random.random((1, 4092, 2)), dtype="float32")
    bbox = np.array(np.random.random((1, 4092, 4)), dtype="float32")
    anchors = np.array(np.random.random((1, 4092, 4)), dtype="float32")
    conf = Conf()
    P = Proposals(conf, batch_size=1, DEBUG=True)
    out = P.run(probs, bbox, anchors)                     # host numpy in, like the reference's feed_dict
    assert tuple(out.shape) == (1, 1000, 4)
    _check_proposals(P, probs, bbox, anchors, conf)
    g = P.get_proposal_graph()
    assert set(g) == {"rpn_class_probs", "rpn_bbox", "input_anchors", "proposals"}


@pytest.mark.parametrize("training", [False, True])
def test_proposals_coco_shape(training):
    """BASELINE config 2: 1024^2, 261,888 anchors, 6000 pre-NMS -> 1000 (2000 training), batch 2."""
    from objectdetection_b200 import Proposals, utils
    conf = Conf()
    rs = np.random.RandomState(1234)
    shapes = utils.get_resnet_stage_shapes(conf, conf.IMAGE_SHAPE)
    anchors = oracle.gen_anchors(conf.IMAGE_SHAPE, 2, conf.RPN_ANCHOR_SCALES, conf.RPN_ANCHOR_RATIOS, shapes,
                                 conf.RESNET_STRIDES, conf.RPN_ANCHOR_STRIDE)
    probs, bbox = _synth.rpn_outputs(rs, 2, anchors.shape[1])
    P = Proposals(conf, 2, cu(probs), cu(bbox), cu(anchors), training=training, DEBUG=True)
    want = _check_proposals(P, probs, bbox, anchors, conf, training)
    # same result when the decode kernel regenerates the anchors from their index (fused anchor generation)
    spec = utils.anchor_spec(conf.IMAGE_SHAPE, conf.RPN_ANCHOR_SCALES, conf.RPN_ANCHOR_RATIOS, shapes,
                             conf.RESNET_STRIDES, conf.RPN_ANCHOR_STRIDE)
    P2 = Proposals(conf, 2, cu(probs), cu(bbox), None, training=training, anchor_spec=spec)
    assert_bits(host(P2.get_proposals()), want, "proposals (fused anchors)")
    # properties: inside [0,1], zero rows only at the tail
    p = host(P.get_proposals())
    assert p.min() >= 0 and p.max() <= 1
    nz = np.abs(p).sum(-1) != 0
    for b in range(2):
        assert not nz[b, int(host(P.num_kept)[b]):].any()


def test_proposals_from_rpn_level_outputs():
    """SURVEY 8(f)3: the layer fed by the RPN head's per-level conv outputs (rpn.py:50-67, training.py:146-166):
    bit-identical to flattening them on the host (oracle.rpn_levels_to_flat) and running the [B,A,.] layer."""
    from objectdetection_b200 import Proposals, utils
    for conf, B, training in ((Conf(), 2, False), (ShapesConfig(), 3, True)):
        rs = np.random.RandomState(77)
        shapes = utils.get_resnet_stage_shapes(conf, conf.IMAGE_SHAPE)
        na = len(conf.RPN_ANCHOR_RATIOS)
        logits = [rs.normal(0, 2, (B, int(h), int(w), 2 * na)).astype(f32) for h, w in shapes]
        bbox = [rs.normal(0, 1, (B, int(h), int(w), 4 * na)).astype(f32) for h, w in shapes]
        probs, flat = oracle.rpn_levels_to_flat(logits, bbox)
        anchors = oracle.gen_anchors(conf.IMAGE_SHAPE, B, conf.RPN_ANCHOR_SCALES, conf.RPN_ANCHOR_RATIOS, shapes,
                                     conf.RESNET_STRIDES, conf.RPN_ANCHOR_STRIDE)
        assert probs.shape[1] == anchors.shape[1]
        P = Proposals(conf, B, training=training, DEBUG=True)
        P.run_levels([cu(t) for t in logits], [cu(t) for t in bbox], cu(anchors))
        want = _check_proposals(P, probs, flat, anchors, conf, training)
        # the [B,A,.] entry point on the flattened tensors gives the same bits; so does regenerating the anchors
        P1 = Proposals(conf, B, cu(probs), cu(flat), cu(anchors), training=training)
        assert_bits(host(P1.get_proposals()), want, "flat entry point")
        spec = utils.anchor_spec(conf.IMAGE_SHAPE, conf.RPN_ANCHOR_SCALES, conf.RPN_ANCHOR_RATIOS, shapes,
                                 conf.RESNET_STRIDES, conf.RPN_ANCHOR_STRIDE)
        P2 = Proposals(conf, B, training=training, anchor_spec=spec)
        assert_bits(host(P2.run_levels(logits, bbox)), want, "levels + fused anchors (host inputs)")
    with pytest.raises(ValueError):
        P2.run_levels(logits[:2], bbox)
    with pytest.raises(ValueError):                                    # bbox channel count must be twice the logits'
        P2.run_levels(logits, [b[..., :4] for b in bbox])


def test_proposals_toy_config_with_padding():
    """BASELINE config 1 (shapes.py): 128x128, 4092 anchors, K = min(6000, 4092); low threshold -> zero padded rows."""
    from objectdetection_b200 import Proposals, utils
    conf = ShapesConfig()
    conf.RPN_NMS_THRESHOLD = 0.05
    rs = np.random.RandomState(5)
    shapes = utils.get_resnet_stage_shapes(conf, conf.IMAGE_SHAPE)
    anchors = oracle.gen_anchors(conf.IMAGE_SHAPE, 8, conf.RPN_ANCHOR_SCALES, conf.RPN_ANCHOR_RATIOS, shapes,
                                 conf.RESNET_STRIDES, 1)
    probs, bbox = _synth.rpn_outputs(rs, 8, 4092)
    P = Proposals(conf, 8, cu(probs), cu(bbox), cu(anchors), DEBUG=True)
    want = _check_proposals(P, probs, bbox, anchors, conf)
    assert (np.abs(want).sum(-1) == 0).any()


# ------------------------------------------------------------------ PyramidROIAlign
def _roi_align_check(fmaps, props, image, pool):
    from objectdetection_b200 import MaskRCNN
    m = MaskRCNN(image_shape=[image, image, 3], pool_shape=pool, num_classes=4, levels=[2, 3, 4, 5],
                 proposals=cu(props), feature_maps=[cu(f) for f in fmaps], type='keras', DEBUG=True)
    got = host(m.get_pooled_rois())
    want, wlv = oracle.pyramid_roi_align(fmaps, props, image, image, pool[0], pool[1])
    assert got.shape == want.shape == (1, props.shape[0] * props.shape[1], pool[0], pool[1], fmaps[0].shape[-1])
    assert np.array_equal(host(m.debug_outputs()[0]), wlv)                      # roi_level bit-exact
    assert np.allclose(got, want, rtol=1e-4, atol=0)                             # north-star tolerance
    frac = (got.view(np.uint32) == want.view(np.uint32)).mean()
    assert frac == 1.0, f"only {frac:.6f} of the pooled values are bit-identical"
    return got


@pytest.mark.parametrize("pool", [[7, 7], [14, 14]])
def test_roi_pooling_debug_recipe(pool):
    """maskrcnn.py:327-345: seed 255, P2..P5 (2,{256,128,64,32}^2,256), proposals (2,1000,4) uniform."""
    np.random.seed(255)
    fmaps = [np.array(np.random.random((2, s, s, 256)), dtype="float32") for s in (256, 128, 64, 32)]
    props = np.array(np.random.random((2, 1000, 4)), dtype="float32")
    _roi_align_check(fmaps, props, 1024, pool)


def test_roi_pooling_realistic_rois_and_degenerates():
    rs = np.random.RandomState(1234)
    fmaps = _synth.pyramid(rs, 2, D=64)
    props = _synth.rois_log_uniform(rs, 2, 400)
    props[1, 350:] = 0                                                        # zero padded proposals -> level 2
    props[0, 0] = [0, 0, 1, 1]
    props[0, 1] = [0.3, 0.3, 0.3, 0.3]
    props[0, 2] = [0.25, 0.5, 1.0, 1.0]                                       # touches the far edge
    props[0, 3] = [-0.1, -0.2, 0.4, 0.5]                                      # partly outside -> extrapolation 0
    props[0, 4] = [0.5, 0.5, 1.2, 1.3]
    for pool in ([7, 7], [14, 14], [1, 1], [3, 5]):
        got = _roi_align_check(fmaps, props, 1024, pool)
    lv = oracle.roi_level(props, 1024, 1024)
    assert set(np.unique(lv)) == {2, 3, 4, 5}


@pytest.mark.parametrize("pool", [[7, 7], [14, 14], [1, 1], [3, 5], [16, 16], [5, 14], [14, 2]])
def test_roi_pooling_d256_rows_kernel_edge_cases(pool):
    """D = 256 goes through the TMA-staged separable kernel (crop_rows_kernel): up-sampled, down-sampled, thin, flipped,
    NaN, zero-area, out-of-image and whole-image ROIs on a small pyramid, every pooled value bit-identical."""
    rs = np.random.RandomState(4321 + pool[0])
    fmaps = [rs.random_sample((2, s, s, 256)).astype(f32) for s in (64, 32, 16, 8)]
    props = _synth.rois_with_edge_cases(rs, 2, 160)
    _roi_align_check(fmaps, props, 1024, pool)
    _roi_align_check(fmaps, props, 1024, pool)                                # again: the ticket counter was left zeroed
    from objectdetection_b200 import _lib
    torch.cuda.synchronize()
    assert all(int(w[:256].count_nonzero()) == 0 for w in _lib._zero_ws.values())   # the ticket counters; the rest is scratch


@pytest.mark.parametrize("pool,n", [([14, 14], 700), ([7, 7], 700), ([14, 14], 4500)])
def test_roi_pooling_processing_order(pool, n):
    """>= 512 ROIs: roi_order_kernel buckets the ROIs by (approximate level, y band) and both ROIAlign kernels walk them in
    that order; NaN / zero / flipped / outside boxes must land in valid buckets and every output row must still be the
    row of ITS ROI. 4500 ROIs per image exceed the pre-pass's capacity (4096): index order, same results."""
    rs = np.random.RandomState(77 + n + pool[0])
    fmaps = [rs.random_sample((2, s, s, 256)).astype(f32) for s in (64, 32, 16, 8)]
    props = _synth.rois_log_uniform(rs, 2, n, lo=4, hi=900)
    props[0, 3] = [np.nan, 0.1, 0.5, 0.6]
    props[0, 4] = [0.1, np.nan, np.nan, 0.6]
    props[0, 5] = [0.9, 0.1, 0.2, 0.8]                                        # flipped
    props[0, 6] = 0                                                           # zero area at the origin
    props[0, 7] = [1.5, 1.5, 2.0, 2.0]                                        # outside
    props[0, 8] = [-3.0, -3.0, -2.0, -2.0]                                    # negative centre
    props[0, 9] = [np.inf, 0.0, np.inf, 1.0]
    props[1, n - 50:] = 0                                                     # zero padding
    _roi_align_check(fmaps, props, 1024, pool)


def test_roi_pooling_without_workspace_static_round_robin():
    """od_pyramid_roi_align_forward (no workspace): the persistent CTAs walk the ROIs in a fixed round robin, in index
    order, without the order pre-pass - same bits."""
    import ctypes
    from objectdetection_b200 import _lib
    rs = np.random.RandomState(31)
    fmaps = [rs.random_sample((2, s, s, 256)).astype(f32) for s in (64, 32, 16, 8)]
    props = _synth.rois_log_uniform(rs, 2, 400, lo=4, hi=900)
    want, wlv = oracle.pyramid_roi_align(fmaps, props, 1024, 1024, 14, 14)
    L = _lib.lib()
    dl = _lib.DL()
    fm = [cu(f) for f in fmaps]
    rois = cu(props)
    out = torch.empty((1, 800, 14, 14, 256), dtype=torch.float32, device="cuda")
    lv = torch.empty((2, 400), dtype=torch.int32, device="cuda")
    ptrs = (ctypes.c_void_p * 4)(*[dl(f) for f in fm])
    _lib.check(L.od_pyramid_roi_align_forward(ptrs, 4, 2, dl(rois), 1024, 1024, 14, 14, dl(out), dl(lv),
                                              _lib.stream_ptr(rois.device)), "od_pyramid_roi_align_forward")
    assert_bits(host(out), want, "pooled (static round robin)")
    assert np.array_equal(host(lv), wlv)


@pytest.mark.parametrize("pool", [[14, 14], [7, 7]])
def test_roi_pooling_caller_supplied_order(pool):
    """roi_processing_order computed once and passed to the pooling call: same bits as the call's own pre-pass; the order
    is a permutation; a corrupted order (out-of-range and duplicated entries) skips / repeats rows without touching
    anything else - the rows of skipped ROIs keep their previous contents."""
    from objectdetection_b200.maskrcnn import pyramid_roi_align, roi_processing_order
    rs = np.random.RandomState(5 + pool[0])
    fmaps = [rs.random_sample((2, s, s, 256)).astype(f32) for s in (64, 32, 16, 8)]
    props = _synth.rois_log_uniform(rs, 2, 600, lo=4, hi=900)
    props[1, 590:] = 0
    want, _ = oracle.pyramid_roi_align(fmaps, props, 1024, 1024, pool[0], pool[1])
    fm, pr = [cu(f) for f in fmaps], cu(props)
    order = roi_processing_order(pr, [1024, 1024, 3])
    assert sorted(host(order).tolist()) == list(range(1200))
    got = host(pyramid_roi_align(fm, pr, [1024, 1024, 3], pool, order=order))
    assert_bits(got, want, "pooled with a caller-supplied order")
    mode = int(os.environ.get("OD_ROI_ORDER", "2"))      # developer switch of the library: 0 = orders are ignored,
    if mode == 0 or (mode == 1 and pool[0] < 10):        # 1 = only the row-ring kernel (pool >= 10) walks an order
        return
    bad = host(order).copy()
    skipped = [int(bad[3]), int(bad[700])]
    bad[3], bad[700] = -1, 5000                       # two ROIs are never visited ...
    bad[10] = bad[11]                                 # ... one is visited twice, one (bad[10]'s old ROI) not at all
    skipped.append(int(host(order)[10]))
    out = torch.full((1, 1200, pool[0], pool[1], 256), -7.0, dtype=torch.float32, device="cuda")
    got2 = host(pyramid_roi_align(fm, pr, [1024, 1024, 3], pool, out=out, order=cu(bad.astype(np.int32))))
    keep = np.ones(1200, bool)
    keep[skipped] = False
    assert_bits(got2[0, keep], want[0, keep], "rows of the visited ROIs")
    assert (got2[0, ~keep] == -7.0).all(), "rows of skipped ROIs must stay untouched"


def test_crop_and_resize_d256_rows_kernel():
    """tf.image.crop_and_resize entry (explicit box_ind, extrapolation value, skipped crops) on the D = 256 path."""
    from objectdetection_b200.maskrcnn import crop_and_resize
    rs = np.random.RandomState(12)
    img = rs.random_sample((3, 19, 23, 256)).astype(f32)
    boxes = np.concatenate([np.array([[0, 0, 1, 1], [0.1, 0.2, 0.7, 0.9], [0.3, 0.3, 0.3, 0.3], [-0.2, -0.1, 0.5, 0.5],
                                      [0.5, 0.5, 1.3, 1.2], [0.9, 0.8, 0.1, 0.2], [0, 0, 0, 0], [0.25, 0.5, 0.75, 1.0]], f32),
                            _synth.random_boxes(rs, 24, flip=True)])
    bi = rs.randint(0, 3, boxes.shape[0]).astype(np.int32)
    bi[7], bi[9] = 5, -1                                                      # out of range: crop left untouched
    for crop in ((7, 7), (14, 14), (1, 1), (1, 3), (16, 9)):
        out0 = np.full((boxes.shape[0], crop[0], crop[1], 256), -7.0, f32)
        got = host(crop_and_resize(cu(img), cu(boxes), cu(bi), crop, extrapolation_value=0.5, out=cu(out0)))
        want = oracle.crop_and_resize(img, boxes, bi, crop[0], crop[1], extrapolation=0.5, out=out0.copy())
        assert_bits(got, want, f"crop {crop}")
        assert (got[7] == -7.0).all() and (got[9] == -7.0).all()


def test_roi_align_properties_full_size():
    """Size-independent properties at the BASELINE size (2 x 1000 ROIs x 7x7 x 256): linearity in the feature maps
    and exactness on a constant pyramid."""
    from objectdetection_b200.maskrcnn import pyramid_roi_align
    rs = np.random.RandomState(7)
    props = cu(_synth.rois_log_uniform(rs, 2, 1000))
    f1 = [torch.rand((2, s, s, 256), device="cuda") for s in (256, 128, 64, 32)]
    f2 = [torch.rand((2, s, s, 256), device="cuda") for s in (256, 128, 64, 32)]
    a = pyramid_roi_align(f1, props, [1024, 1024], [7, 7])
    b = pyramid_roi_align(f2, props, [1024, 1024], [7, 7])
    c = pyramid_roi_align([2 * x + y for x, y in zip(f1, f2)], props, [1024, 1024], [7, 7])
    assert torch.allclose(c, 2 * a + b, rtol=1e-4, atol=1e-5)
    const = pyramid_roi_align([torch.full_like(x, 3.25) for x in f1], props, [1024, 1024], [7, 7])
    assert bool(((const == 3.25) | (const == 0)).all()) and float((const == 3.25).float().mean()) > 0.99


def test_crop_and_resize_generic():
    from objectdetection_b200.maskrcnn import crop_and_resize
    rs = np.random.RandomState(2)
    img = rs.random_sample((2, 9, 11, 8)).astype(f32)
    boxes = np.array([[0, 0, 1, 1], [0.1, 0.2, 0.7, 0.9], [0.3, 0.3, 0.3, 0.3], [-0.2, -0.1, 0.5, 0.5],
                      [0.5, 0.5, 1.3, 1.2], [0.9, 0.8, 0.1, 0.2], [0, 0, 0, 0], [0.25, 0.5, 0.75, 1.0]], f32)
    bi = np.array([0, 1, 0, 1, 0, 1, 0, 5], np.int32)
    for crop in ((7, 7), (14, 14), (1, 1), (1, 3), (2, 2)):
        got = host(crop_and_resize(cu(img), cu(boxes), cu(bi), crop, extrapolation_value=0.5))
        want = oracle.crop_and_resize(img, boxes, bi, crop[0], crop[1], extrapolation=0.5)
        assert_bits(got, want, f"crop {crop}")


# ------------------------------------------------------------------ DetectionTargetLayer
def _check_targets(conf, props, cls, gt, pp, pn):
    from objectdetection_b200 import BuildDetectionTargets
    B = props.shape[0]
    t = BuildDetectionTargets(conf, cu(props), cu(cls), cu(gt), DEBUG=True, perm_pos=cu(pp), perm_neg=cu(pn))
    rois, rcls, deltas = (host(x) for x in t.get_target_rois())
    d = {k: host(v) for k, v in t.debug_raw.items()}
    R = conf.MRCNN_TRAIN_ROIS_PER_IMAGE
    assert rois.shape == (B, R, 4) and rcls.shape == (B, R) and deltas.shape == (B, R, 4)
    for b in range(B):
        w_rois, w_cls, w_deltas, wd = oracle.detection_targets(props[b], cls[b], gt[b], pp[b], pn[b], R, conf.BBOX_STD_DEV)
        assert np.array_equal(d["counts"][b], wd["counts"]), (b, d["counts"][b], wd["counts"])
        n_prop, n_gt = wd["counts"][:2]
        assert np.array_equal(d["pos_indices"][b], wd["pos_indices"])            # bit-exact index lists
        assert np.array_equal(d["neg_indices"][b], wd["neg_indices"])
        assert np.array_equal(d["sampled_pos"][b], wd["sampled_pos"])
        assert np.array_equal(d["sampled_neg"][b], wd["sampled_neg"])
        assert np.array_equal(d["gt_assignment"][b], wd["gt_assignment"])
        assert_bits(d["iou"][b][:n_prop, :n_gt], wd["iou"][:n_prop, :n_gt], "iou")
        assert_bits(d["roi_iou_max"][b][:n_prop], wd["roi_iou_max"][:n_prop], "iou max")
        assert_bits(rois[b], w_rois, "rois")
        assert np.array_equal(rcls[b], w_cls[0])
        assert_bits(deltas[b], w_deltas, "deltas")
        assert np.allclose(deltas[b], w_deltas, rtol=1e-5, equal_nan=True)
    return d


def test_detection_targets_training_config():
    """BASELINE config 3: 2000 proposals, 100 GT, 200 sampled ROIs (33% positive), batch 8."""
    rs = np.random.RandomState(77)
    conf = Conf()
    d = _check_targets(conf, *_synth.target_inputs(rs, 8, 2000, 100))
    assert (d["counts"][:, 4] > 0).all() and (d["counts"][:, 4] <= 66).all()


@pytest.mark.parametrize("mini", [True, False])
def test_detection_mask_targets(mini):
    """28x28 mask-target crops (north-star extension): blob masks, mini-mask and full-image variants, batch 3."""
    from objectdetection_b200 import BuildDetectionTargets
    rs = np.random.RandomState(11)

    class C(Conf):
        USE_MINI_MASK = mini
    conf = C()
    B, N, G, M = 3, 600, 20, 56
    props, cls, gt, pp, pn = _synth.target_inputs(rs, B, N, G, n_pad=100)
    masks = np.zeros((B, M, M, G), f32)                      # reference layout [B,Mh,Mw,G]
    yy, xx = np.mgrid[0:M, 0:M]
    for b in range(B):
        for g in range(G):
            cy, cx, r = rs.uniform(10, 46), rs.uniform(10, 46), rs.uniform(6, 25)
            masks[b, :, :, g] = ((yy - cy) ** 2 + (xx - cx) ** 2 < r * r).astype(f32)
    t = BuildDetectionTargets(conf, cu(props), cu(cls), cu(gt), DEBUG=True, perm_pos=cu(pp), perm_neg=cu(pn),
                              gt_masks=cu(masks))
    got = host(t.get_target_masks())
    rois = host(t.get_target_rois()[0])
    R = conf.MRCNN_TRAIN_ROIS_PER_IMAGE
    assert got.shape == (B, R, 28, 28)
    n_pos_total = 0
    for b in range(B):
        w_rois, _, _, wd = oracle.detection_targets(props[b], cls[b], gt[b], pp[b], pn[b], R, conf.BBOX_STD_DEV)
        assert_bits(rois[b], w_rois, "rois")
        want = oracle.mask_targets(w_rois, cls[b], gt[b], masks[b], wd, (28, 28), mini)
        assert np.array_equal(got[b], want), (b, np.abs(got[b] - want).sum())       # {0,1} values: exact
        n_pos_total += int(wd["counts"][4])
        assert not got[b, int(wd["counts"][4]):].any()
    assert n_pos_total > 0 and got.any() and set(np.unique(got)) <= {0.0, 1.0}


def test_detection_targets_edge_cases():
    rs = np.random.RandomState(3)
    conf = ShapesConfig()
    props, cls, gt, pp, pn = _synth.target_inputs(rs, 4, 300, 10, n_pad=40)
    cls[1] = 0                                   # image without GT -> all zero targets
    props[2, 5] = 0                              # a zero row in the middle: compacted indices hit the un-compacted tensor
    props[3, :250] = 0                           # almost everything padded
    d = _check_targets(conf, props, cls, gt, pp, pn)
    assert d["counts"][1, 4] == 0 and d["counts"][1, 5] == 0


def test_detection_targets_per_image_signature():
    """The reference calls BuildDetectionTargets per image (training.py:71-73): [N,4], [G], [G,4] -> [R,4], [1,R], [R,4]."""
    from objectdetection_b200 import BuildDetectionTargets
    rs = np.random.RandomState(8)
    conf = ShapesConfig()
    props, cls, gt, pp, pn = _synth.target_inputs(rs, 1, 120, 6, n_pad=20)
    t = BuildDetectionTargets(conf, props[0], cls[0], gt[0], perm_pos=pp[0], perm_neg=pn[0])
    rois, rcls, deltas = t.get_target_rois()
    assert tuple(rois.shape) == (32, 4) and tuple(rcls.shape) == (1, 32) and tuple(deltas.shape) == (32, 4)
    w_rois, w_cls, w_deltas, _ = oracle.detection_targets(props[0], cls[0], gt[0], pp[0], pn[0], 32, conf.BBOX_STD_DEV)
    assert_bits(host(rois), w_rois, "rois")
    assert np.array_equal(host(rcls), w_cls)
    # unseeded path: counts only
    t2 = BuildDetectionTargets(conf, props[0], cls[0], gt[0], DEBUG=True)
    assert int(t2.debug_raw["counts"][0, 4]) == int((w_cls > 0).sum())
    assert int(t2.debug_outputs()["pos_count"]) == int((w_cls > 0).sum()) and len(t2.debug_outputs()) == 21


# ------------------------------------------------------------------ DetectionLayer
def _check_detection(conf, window_px, image_shape, props, probs, bbox):
    from objectdetection_b200 import DetectionLayer
    D = DetectionLayer(conf, image_shape, props.shape[0], window_px, cu(props), cu(probs), cu(bbox), DEBUG=True)
    win = oracle.norm_boxes(window_px, image_shape[:2])
    want, wd = oracle.detection_forward(props, probs, bbox, win, conf.BBOX_STD_DEV, conf.DETECTION_MIN_THRESHOLD,
                                        conf.DETECTION_NMS_THRESHOLD, conf.DETECTION_POST_NMS_INSTANCES, debug=True)
    assert np.array_equal(host(D.class_ids), wd["class_ids"])
    assert_bits(host(D.class_scores), wd["class_scores"], "class_scores")
    assert_bits(host(D.refined_proposals), wd["refined_proposals"], "refined")
    assert np.allclose(host(D.refined_proposals), wd["refined_proposals"], rtol=1e-5, equal_nan=True)
    assert_bits(host(D.clipped_proposals), wd["clipped_proposals"], "clipped")
    assert np.array_equal(host(D.keep_mask), wd["keep_mask"])
    assert np.array_equal(host(D.nms_keep_mask), wd["nms_keep_mask"])
    got = host(D.get_detections())
    assert_bits(got, want, "detections")
    return got


def test_detection_debug_recipe():
    """detection.py:285-310: seed 863, (1,8,4) / (1,8,4) / (1,8,4,4), window [131,0,893,1024]."""
    np.random.seed(863)
    props = np.array(np.random.random((1, 8, 4)), dtype="float32")
    probs = np.array(np.random.random((1, 8, 4)), dtype="float32")
    bbox = np.array(np.random.random((1, 8, 4, 4)), dtype="float32")
    det = _check_detection(Conf(), np.array([[131, 0, 893, 1024]], "int32"), [1024, 1024, 3], props, probs, bbox)
    assert det.shape == (1, 100, 6)


def test_detection_coco_shape():
    """BASELINE config 2: [2,1000,81] head outputs, window [131,0,893,1024]."""
    rs = np.random.RandomState(1234)
    props = _synth.rois_log_uniform(rs, 2, 1000)
    props[1, 900:] = 0
    probs, bbox = _synth.head_outputs(rs, 2, 1000, 81)
    win = np.array([[131, 0, 893, 1024], [0, 0, 1024, 1024]], "int32")
    det = _check_detection(Conf(), win, [1024, 1024, 3], props, probs, bbox)
    assert (det[:, :, 4] > 0).sum() > 50
    from objectdetection_b200.detection import unmold_detection
    b, c, s = unmold_detection((600, 800, 3), (1024, 1024, 3), det[0], win[0])
    wb, wc, ws_ = oracle.unmold_detection((600, 800, 3), (1024, 1024, 3), det[0], win[0])
    assert np.array_equal(b, wb) and np.array_equal(c, wc) and np.array_equal(s, ws_)


def test_detection_ties_caps_and_empty():
    rs = np.random.RandomState(9)
    B, N, C = 2, 400, 6
    props = _synth.random_boxes(rs, B * N).reshape(B, N, 4)
    probs, bbox = _synth.head_outputs(rs, B, N, C, boosted=0.9)
    probs = (np.round(probs * 64) / 64).astype(f32)                 # quantised -> score ties
    conf = Conf()
    conf.DETECTION_POST_NMS_INSTANCES = 40                          # per-class cap and final cap both bind
    win = np.array([[100, 0, 900, 1024], [0, 0, 1024, 1024]], "int32")
    det = _check_detection(conf, win, [1024, 1024, 3], props, probs, bbox)
    assert np.all(np.diff(det[:, :, 5], axis=1) <= 0)
    empty = _check_detection(conf, win, [1024, 1024, 3], props, np.full_like(probs, 1.0 / C), bbox)
    assert not empty.any()


# ------------------------------------------------------------------ Faster R-CNN
def test_frcnn_proposals_and_roi_pool(golden):
    """BASELINE config 4: 600x1000, stride 16 (38x63 -> 21,546 anchors), 12000 -> 2000; thr 0.7 and the reference's 0.2."""
    from objectdetection_b200 import fasterrcnn
    rs = np.random.RandomState(9)
    h, w, na = 38, 63, 9
    probs = rs.random_sample((1, h, w, 2 * na))
    bbox = rs.normal(0, 0.5, size=(1, h, w, 4 * na))
    for thr in (0.7, 0.2):
        P = fasterrcnn.Proposals('train', probs, bbox, image_shape=(600, 1000, 3), nms_threshold=thr)
        got = host(P.get_proposals())
        want = oracle.frcnn_proposals(probs, bbox, 600, 1000, 12000, 2000, thr)
        assert got.shape == want.shape and np.all(got[:, 0] == 0)
        # every kept box, in visiting order, bit for bit (fp64 decode rounded once to f32): equal rows in equal order also
        # pin the NMS keep sequence, which the fp32 screening pass in frcnn.cu must not change
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    # float32 inputs take the radix-select top-k instead of the 128-bit rank sort: same visiting order, ties (scores
    # quantised to 3 decimals) go to the lower index, filtered-out boxes never enter
    p32 = np.round(probs, 3).astype(f32)
    b32 = bbox.astype(f32)
    for thr, pre in ((0.7, 12000), (0.2, 3000)):
        P = fasterrcnn.Proposals('train', cu(p32), cu(b32), image_shape=(600, 1000, 3), nms_threshold=thr, pre_nms_top_n=pre)
        got32 = host(P.get_proposals())
        want32 = oracle.frcnn_proposals(p32.astype(np.float64), b32.astype(np.float64), 600, 1000, pre, 2000, thr)
        assert got32.shape == want32.shape
        assert np.array_equal(got32.view(np.uint32), want32.view(np.uint32))
    assert np.array_equal(fasterrcnn.get_anchors(), golden["frcnn_base_anchors"])
    # golden: the reference's own decode -> clip -> filter -> NMS on the small 6x9 case
    gp = np.zeros((1, 6, 9, 18))
    gp[0, :, :, :9] = golden["frcnn_scores_all"].reshape(6, 9, 9)
    gb = golden["frcnn_deltas"].reshape(1, 6, 9, 36)
    for thr in (0.2, 0.7):
        P = fasterrcnn.Proposals('test', gp, gb, image_shape=(96, 144, 3), nms_threshold=thr, pre_nms_top_n=10 ** 9 // 2,
                                 post_nms_top_n=50)
        ref = golden[f"frcnn_nms_out_thr{int(thr * 10)}"].astype(f32)
        assert np.array_equal(host(P.get_proposals())[:, 1:], ref)    # the reference's own run, rounded to f32
    fmap = rs.random_sample((1, h, w, 512)).astype(f32)
    rois = want[:300]   # the thr=0.2 run keeps ~200 boxes of this input
    assert rois.shape[0] > 100
    pooled = host(fasterrcnn.roi_pool(cu(fmap), cu(rois), (600, 1000, 3)))
    wp = oracle.roi_pool(fmap, rois, 600.0, 1000.0)
    assert pooled.shape == (rois.shape[0], 7, 7, 512)
    assert_bits(pooled, wp, "roi_pool")


# ------------------------------------------------------------------ device unmold (SURVEY §8f)
def test_unmold_detections_on_device(golden):
    """od_unmold_detections (batched) and the reference-shaped single-image wrapper over it vs the oracle's numpy
    restatement (pinned by the reference's own numpy code in test_abi.test_oracle_unmold_golden) on synthetic
    detections, plus zero-area / empty / full edge rows."""
    from objectdetection_b200.detection import unmold_detection, unmold_detections_batch
    rs = np.random.RandomState(31)
    B, M = 5, 100
    det = np.zeros((B, M, 6), f32)
    for b, n in enumerate([37, 0, 100, 5, 64]):
        y1 = rs.uniform(0.13, 0.8, n); x1 = rs.uniform(0.0, 0.9, n)
        det[b, :n, 0], det[b, :n, 1] = y1, x1
        det[b, :n, 2], det[b, :n, 3] = y1 + rs.uniform(0, 0.07, n), x1 + rs.uniform(0, 0.1, n)
        det[b, :n, 4] = rs.randint(1, 81, n)
        det[b, :n, 5] = rs.uniform(0.7, 1, n)
    det[0, 3, 2:4] = det[0, 3, 0:2]                      # zero-size row: 1 px after the +1 shift of denorm_boxes -> kept
    det[0, 7, 3] = det[0, 7, 1] - 0.01                   # flipped in x -> negative area -> dropped
    det[3, 1, 2] = det[3, 1, 0] - 0.01                   # flipped -> negative area -> dropped
    windows = np.array([[131, 0, 893, 1024], [0, 0, 1024, 1024], [131, 0, 893, 1024], [0, 100, 1024, 924], [131, 0, 893, 1024]])
    shapes = np.array([[480, 640, 3], [1024, 1024, 3], [375, 500, 3], [600, 600, 3], [720, 1280, 3]])
    boxes, cls, scores, counts = (host(x) for x in unmold_detections_batch(shapes, [1024, 1024, 3], cu(det), windows))
    for b in range(B):
        wb, wc, ws = oracle.unmold_detection(shapes[b], [1024, 1024, 3], det[b], windows[b])
        sb, sc, ss = unmold_detection(shapes[b], [1024, 1024, 3], det[b], windows[b])     # single-image wrapper
        assert np.array_equal(sb, wb) and np.array_equal(sc, wc) and np.array_equal(ss, ws)
        n = counts[b]
        assert n == wb.shape[0]
        assert np.array_equal(boxes[b, :n], wb) and np.array_equal(cls[b, :n], wc) and np.array_equal(scores[b, :n], ws)
        assert not boxes[b, n:].any() and not cls[b, n:].any()
    assert counts.tolist() == [36, 0, 100, 4, 64]


# ------------------------------------------------------------------ RPN targets (SURVEY §8f)
def test_rpn_targets_golden_and_coco_shape():
    """PreprareTrainData.build_rpn_targets: (1) the reference's own outputs (golden, subsampling replayed),
    (2) COCO shape: 261,888 anchors x up to 100 GT boxes, batch 3, against the numpy oracle."""
    import os
    from objectdetection_b200.data_processor import PreprareTrainData
    from objectdetection_b200 import ShapesConfig, config
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_rpn_targets.npz"))

    class Sub(config):
        IMAGE_SHAPE = [256, 256, 3]
        RPN_ANCHOR_SCALES = (16, 32, 64, 128, 256)
        RPN_TRAIN_ANCHORS_PER_IMAGE = 16
    for case, conf in (("toy", ShapesConfig()), ("sub", Sub())):
        P = PreprareTrainData(conf)
        assert np.array_equal(host(P.anchors), g[case + "_anchors"])
        pos, cls, bbox = P.build_rpn_targets(g[case + "_gt"], perm_pos=g[case + "_perm_pos"], perm_neg=g[case + "_perm_neg"])
        assert np.array_equal(host(cls), g[case + "_cls"])                        # labels: bit-exact
        assert np.array_equal(host(pos), g[case + "_pos_anchors"])
        assert np.allclose(host(bbox), g[case + "_bbox"], rtol=1e-13, atol=0)     # fp64 deltas (log may differ by an ulp)
    # COCO shape against the oracle: the reference's limits (100 GT, 256 targets: fused per-GT arg-max), then 300 GT
    # (the per-GT kernel) with 16 targets so that the positives are subsampled too
    class Few(Conf):
        RPN_TRAIN_ANCHORS_PER_IMAGE = 16
    for conf, G, cnt in ((Conf(), 100, [100, 37, 1]), (Few(), 300, [300, 129, 0])):
        P = PreprareTrainData(conf)
        A = P.anchors.shape[0]
        assert A == 261888
        rs = np.random.RandomState(21 + G)
        B, T = 3, conf.RPN_TRAIN_ANCHORS_PER_IMAGE
        anc = host(P.anchors)
        gt = np.zeros((B, G, 4))
        cnt = np.array(cnt, np.int32)
        for b in range(B):
            pick = rs.choice(A, cnt[b], replace=False)
            gt[b, :cnt[b]] = np.round(np.clip(anc[pick] + rs.normal(0, 3, (cnt[b], 4)), 0, 1024))
            bad = (gt[b, :, 2] <= gt[b, :, 0]) | (gt[b, :, 3] <= gt[b, :, 1])
            gt[b, bad] = [100, 100, 164, 164]
        pp = np.stack([rs.permutation(A) for _ in range(B)]).astype(np.int32)
        pn = np.stack([rs.permutation(A) for _ in range(B)]).astype(np.int32)
        pos, cls, bbox, counts = P.build_rpn_targets(gt, perm_pos=pp, perm_neg=pn, gt_count=cnt, return_counts=True)
        pos, cls, bbox, counts = host(pos), host(cls), host(bbox), host(counts)
        for b in range(B):
            w_pos, w_cls, w_bbox, w_counts = oracle.rpn_targets(anc, gt[b, :cnt[b]], pp[b], pn[b], T, conf.RPN_BBOX_STDDEV)
            assert np.array_equal(counts[b], w_counts), (counts[b], w_counts)
            assert np.array_equal(cls[b], w_cls)
            n = w_counts[2]
            assert np.array_equal(pos[b, :n], w_pos) and not pos[b, n:].any()
            assert np.allclose(bbox[b], w_bbox, rtol=1e-13, atol=0)
            assert (cls[b] == 1).sum() <= T // 2 and (cls[b] == 1).sum() + (cls[b] == -1).sum() == T
        if G == 300:
            assert counts[0, 0] > T // 2 and counts[0, 2] == T // 2      # positives were dropped through perm_pos


# ------------------------------------------------------------------ head losses (SURVEY §8f rank 4)
def test_head_losses():
    """Loss.rpn_class_loss / rpn_box_loss / mrcnn_class_loss / mrcnn_box_loss (loss_optimize.py:11-201): forward values
    against the numpy oracle, rtol 1e-6 (fp64 sums of identical fp32 terms; the order of the sums differs)."""
    from objectdetection_b200.loss_optimize import Loss
    from objectdetection_b200.data_processor import PreprareTrainData
    rs = np.random.RandomState(4)
    # (1) COCO shape: labels and targets from the RPN-target builder
    conf = Conf()
    P = PreprareTrainData(conf)
    A, B, T = P.anchors.shape[0], 2, conf.RPN_TRAIN_ANCHORS_PER_IMAGE
    anc = host(P.anchors)
    gt = np.zeros((B, 20, 4))
    for b in range(B):
        gt[b] = np.round(np.clip(anc[rs.choice(A, 20, replace=False)] + rs.normal(0, 3, (20, 4)), 0, 1024))
        bad = (gt[b, :, 2] <= gt[b, :, 0]) | (gt[b, :, 3] <= gt[b, :, 1])
        gt[b, bad] = [100, 100, 164, 164]
    pp = np.stack([rs.permutation(A) for _ in range(B)]).astype(np.int32)
    _, tcls, tbox = P.build_rpn_targets(gt, perm_pos=pp, perm_neg=pp)
    tcls, tbox = host(tcls).reshape(B, A, 1), host(tbox).astype(f32)
    logits = rs.normal(0, 2, (B, A, 2)).astype(f32)
    pred = rs.normal(0, 1.5, (B, A, 4)).astype(f32)
    w_cls, w_box, w_pos = oracle.rpn_losses(tcls, logits, tbox, pred)
    got_cls = Loss.rpn_class_loss(cu(tcls), cu(logits))
    got_pos, got_box = Loss.rpn_box_loss(cu(tbox), cu(pred), cu(tcls), B)
    assert np.isclose(host(got_cls), w_cls, rtol=1e-6) and w_cls > 0
    assert np.isclose(host(got_box), w_box, rtol=1e-6) and w_box > 0
    assert np.array_equal(host(got_pos), w_pos) and w_pos.shape[0] > 0
    c2, b2, _ = Loss.rpn_losses(tcls, logits, tbox, pred)                       # host inputs, one pass for both
    assert host(c2) == host(got_cls) and host(b2) == host(got_box)              # deterministic
    # (2) ragged small case: more positives than target rows in one image, none in the other; then all neutral
    A2, T2 = 2500, 8
    tc = rs.choice([-1, 0, 1], size=(3, A2), p=[.3, .65, .05]).astype(np.int32)
    tc[1][tc[1] == 1] = 0
    lg, tb, pb = rs.normal(0, 2, (3, A2, 2)).astype(f32), rs.normal(0, 1, (3, T2, 4)).astype(f32), rs.normal(0, 1, (3, A2, 4)).astype(f32)
    w = oracle.rpn_losses(tc, lg, tb, pb)
    g = Loss.rpn_losses(tc, lg, tb, pb, want_pos=True)
    assert np.isclose(host(g[0]), w[0], rtol=1e-6) and np.isclose(host(g[1]), w[1], rtol=1e-6)
    assert np.array_equal(host(g[2]), w[2][:g[2].shape[0]]) and g[2].shape[0] == min(w[2].shape[0], 3 * T2)
    g = Loss.rpn_losses(np.zeros_like(tc), lg, tb, pb)
    assert host(g[0]) == 0.0 and host(g[1]) == 0.0
    # (3) detection-head losses: the reference's debug() recipe (loss_optimize.py:209-219) and the COCO training shape
    for Bm, R, C in ((2, 32, 4), (8, 200, 81)):
        ids = np.zeros((Bm, R), np.int32)
        if C == 4:
            ids[0, 2], ids[0, 3], ids[1, 4] = 1, 2, 1
        else:
            ids[:, :66] = rs.randint(1, C, (Bm, 66))
        tb2, pb2 = rs.random_sample((Bm, R, 4)).astype(f32), rs.random_sample((Bm, R, C, 4)).astype(f32)
        pb2[0, 2, ids[0, 2]] = [0.0, 1.0, 0.5, 1e-9]                            # exercises the epsilon clip
        lg2 = rs.normal(0, 2, (Bm, R, C)).astype(f32)
        act = (rs.random_sample((Bm, C)) > 0.3).astype(f32)
        act[:, 0] = 1
        w_pa, w_c, w_b = oracle.mrcnn_losses(ids, lg2, act, tb2, pb2)
        pa, c = Loss.mrcnn_class_loss(cu(ids), cu(lg2), cu(act))
        bl = Loss.mrcnn_box_loss(cu(tb2), cu(pb2), cu(ids), batch_size=Bm)
        assert np.array_equal(host(pa), w_pa)
        assert np.isclose(host(c), w_c, rtol=1e-6) and np.isclose(host(bl), w_b, rtol=1e-6)
        assert host(Loss.mrcnn_box_loss(tb2, pb2, np.zeros_like(ids), batch_size=Bm)) == 0.0


# ------------------------------------------------------------------ error behaviour
def test_errors_are_loud():
    from objectdetection_b200 import _lib
    from objectdetection_b200.proposals import apply_box_deltas, top_k
    with pytest.raises(ValueError):
        apply_box_deltas(cu(np.zeros((1, 4, 4), f32)), cu(np.zeros((1, 5, 4), f32)))
    with pytest.raises(ValueError):
        top_k(cu(np.zeros((1, 4), f32)), 9)
    L = _lib.lib()
    dl = _lib.DL()
    cpu_t = torch.zeros((1, 4, 4))
    rc = L.od_apply_box_deltas(dl(cpu_t), dl(cpu_t), dl(cpu_t), None)
    assert rc == -4 and b"CPU" in L.od_last_error_detail()
