"""bfloat16 head outputs in Proposals, DetectionLayer and the head losses.

A bf16 value is widened to fp32 exactly and everything after the load is the fp32 path, so every output and every DEBUG
intermediate of a call on bf16 tensors must equal, bit for bit, the fp32 call on ``t.float()`` and the oracle on the
widened arrays. The loss sums are compared with the oracle at the tolerance of test_gpu_parity.test_head_losses (their
summation order differs) and with the fp32 call exactly (the kernels' order is fixed).

Inputs are made as bf16 bit patterns (numpy uint16); ``widen`` gives the fp32 values both reference paths are fed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path[:0] = [HERE, ROOT]
import _synth  # noqa: E402

import oracle  # noqa: E402
from objectdetection_b200.config import ShapesConfig, config as Conf  # noqa: E402
from test_gpu_dispatch import assert_launched  # noqa: E402
from test_gpu_parity import _check_proposals, assert_bits, cu, host  # noqa: E402

torch = pytest.importorskip("torch")
f32 = np.float32
gpu = pytest.mark.gpu
F32, BF16 = torch.float32, torch.bfloat16
PAIRS = [(BF16, BF16), (BF16, F32), (F32, BF16)]          # (logits / probs, deltas / boxes); f32-f32 is test_gpu_parity's
IDS = ["bf16-bf16", "bf16-f32", "f32-bf16"]

# bf16 bit patterns of the edge values: +-inf, NaN of both signs with two payloads, -0, subnormals, the largest finite
EDGE_BITS = [0x7F80, 0xFF80, 0x7FC0, 0x7FA5, 0xFFC0, 0xFF93, 0x8000, 0x0001, 0x8005, 0x7F7F, 0xFF7F]


@pytest.fixture(scope="module")
def _cuda():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (there is no CPU path)")


def to_bits(a):
    """fp32 -> the bits of the nearest bf16 (round to nearest even, as torch converts)."""
    return torch.from_numpy(np.ascontiguousarray(a, f32)).to(BF16).view(torch.int16).numpy().view(np.uint16)


def b16(v):
    """The bits of the bf16 nearest to one value."""
    return int(to_bits(np.array([v], f32))[0])


def widen(bits):
    return (np.asarray(bits, np.uint16).astype(np.uint32) << 16).view(f32)


def dev(bits, dt):
    """The bf16 bits as a CUDA tensor of dtype dt (fp32: the widened values)."""
    if dt == BF16:
        return torch.from_numpy(np.ascontiguousarray(bits).view(np.int16)).cuda().view(BF16)
    return cu(widen(bits))


def same(a, b, what):
    assert_bits(host(a), host(b), what)


# ------------------------------------------------------------------ Proposals
def _same_proposals(P, R, what):
    """Every output and DEBUG intermediate of P equals that of the fp32 call R."""
    for name, x, y in zip(("bbox_delta", "ix", "scores", "anchors", "anchor_delta"), P.debug_outputs(), R.debug_outputs()):
        if name == "ix":
            assert torch.equal(x, y), f"{what}: ix"
        else:
            same(x, y, f"{what}: {name}")
    same(P.get_anchors_delta_clipped(), R.get_anchors_delta_clipped(), f"{what}: clipped")
    assert torch.equal(P.keep_idx, R.keep_idx) and torch.equal(P.num_kept, R.num_kept), f"{what}: keep_idx / num_kept"
    same(P.get_proposals(), R.get_proposals(), f"{what}: proposals")


def _levels(conf, B, training, lg_bits, bb_bits, pairs=PAIRS, spec_too=True):
    """run_levels on every dtype pair against the fp32 call and the oracle, with anchors and with anchor_spec."""
    from objectdetection_b200 import Proposals, utils
    shapes = utils.get_resnet_stage_shapes(conf, conf.IMAGE_SHAPE)
    logits, bbox = [widen(t) for t in lg_bits], [widen(t) for t in bb_bits]
    probs, flat = oracle.rpn_levels_to_flat(logits, bbox)
    anchors = oracle.gen_anchors(conf.IMAGE_SHAPE, B, conf.RPN_ANCHOR_SCALES, conf.RPN_ANCHOR_RATIOS, shapes,
                                 conf.RESNET_STRIDES, conf.RPN_ANCHOR_STRIDE)
    spec = utils.anchor_spec(conf.IMAGE_SHAPE, conf.RPN_ANCHOR_SCALES, conf.RPN_ANCHOR_RATIOS, shapes,
                             conf.RESNET_STRIDES, conf.RPN_ANCHOR_STRIDE)
    R = Proposals(conf, B, training=training, DEBUG=True)
    R.run_levels([cu(t) for t in logits], [cu(t) for t in bbox], cu(anchors))
    want = _check_proposals(R, probs, flat, anchors, conf, training)
    RS = Proposals(conf, B, training=training, DEBUG=True, anchor_spec=spec)
    RS.run_levels([cu(t) for t in logits], [cu(t) for t in bbox])
    assert_bits(host(RS.get_proposals()), host(R.get_proposals()), "fp32 call with anchor_spec")
    for (ld, bd), pid in zip(pairs, IDS):
        lg, bb = [dev(t, ld) for t in lg_bits], [dev(t, bd) for t in bb_bits]
        P = Proposals(conf, B, training=training, DEBUG=True)
        P.run_levels(lg, bb, cu(anchors))
        _check_proposals(P, probs, flat, anchors, conf, training)
        _same_proposals(P, R, f"{pid} anchors")
        if spec_too:
            PS = Proposals(conf, B, training=training, DEBUG=True, anchor_spec=spec)
            PS.run_levels(lg, bb)
            _same_proposals(PS, RS, f"{pid} anchor_spec")
    return want


def _level_bits(rs, conf, B, logit_sd=2.0):
    from objectdetection_b200 import utils
    shapes = utils.get_resnet_stage_shapes(conf, conf.IMAGE_SHAPE)
    na = len(conf.RPN_ANCHOR_RATIOS)
    lg = [to_bits(rs.normal(0, logit_sd, (B, int(h), int(w), 2 * na))) for h, w in shapes]
    bb = [to_bits(rs.normal(0, 1, (B, int(h), int(w), 4 * na))) for h, w in shapes]
    return lg, bb


@gpu
@pytest.mark.parametrize("which", ["coco", "shapes-training"])
def test_run_levels_bf16(_cuda, which):
    """COCO (B = 2, 261,888 anchors) and ShapesConfig (B = 3, training): the three dtype pairs, anchors and anchor_spec,
    every DEBUG intermediate."""
    conf, B, training = (Conf(), 2, False) if which == "coco" else (ShapesConfig(), 3, True)
    rs = np.random.RandomState(77)
    _levels(conf, B, training, *_level_bits(rs, conf, B))


@gpu
def test_run_flat_fp32_probs_bf16_deltas(_cuda):
    """run() with fp32 [B,A,2] probabilities and bf16 [B,A,4] deltas at the COCO shape."""
    from objectdetection_b200 import Proposals, utils
    conf = Conf()
    rs = np.random.RandomState(1234)
    shapes = utils.get_resnet_stage_shapes(conf, conf.IMAGE_SHAPE)
    anchors = oracle.gen_anchors(conf.IMAGE_SHAPE, 2, conf.RPN_ANCHOR_SCALES, conf.RPN_ANCHOR_RATIOS, shapes,
                                 conf.RESNET_STRIDES, conf.RPN_ANCHOR_STRIDE)
    probs, bbox = _synth.rpn_outputs(rs, 2, anchors.shape[1])
    bits = to_bits(bbox)
    for training in (False, True):
        R = Proposals(conf, 2, cu(probs), cu(widen(bits)), cu(anchors), training=training, DEBUG=True)
        _check_proposals(R, probs, widen(bits), anchors, conf, training)
        t = dev(bits, BF16)
        P = Proposals(conf, 2, cu(probs), t, cu(anchors), training=training, DEBUG=True)
        _check_proposals(P, probs, widen(bits), anchors, conf, training)
        _same_proposals(P, R, f"flat bf16 deltas training={training}")
        assert P.get_proposal_graph()["rpn_bbox"] is t          # stored as passed, no fp32 copy


@gpu
def test_run_levels_heavy_ties(_cuda):
    """bf16 logits drawn from a handful of values: thousands of anchors share the 6000th score."""
    conf = Conf()
    rs = np.random.RandomState(5)
    lg, bb = _level_bits(rs, conf, 2)
    lg = [to_bits(rs.choice(np.array([-2.0, -0.5, 0.0, 0.75, 1.5], f32), size=t.shape)) for t in lg]
    want = _levels(conf, 2, False, lg, bb, spec_too=False)
    assert want.shape == (2, 1000, 4)
    # the 6000th score is tied many times over
    probs, _ = oracle.rpn_levels_to_flat([widen(t) for t in lg], [widen(t) for t in bb])
    fg = probs[0, :, 1]
    kth = np.sort(fg)[::-1][5999]
    assert (fg == kth).sum() > 1000


@gpu
def test_run_levels_edge_values(_cuda):
    """+-inf, NaN of both signs with two payloads, -0, bf16 subnormals and the largest finite bf16 (exp overflows in the
    decode), in logits and deltas, at the first and at a later anchor of a level."""
    conf = ShapesConfig()
    rs = np.random.RandomState(2024)
    B = 2
    lg, bb = _level_bits(rs, conf, B)
    for lvl, start in ((0, 0), (0, 700), (3, 5)):
        pairs = lg[lvl].reshape(B, -1, 2)
        rows = bb[lvl].reshape(B, -1, 4)
        for k, e in enumerate(EDGE_BITS):
            j = start + k
            pairs[0, j] = [e, e] if k % 2 else [b16(0.0), e]       # both, or fg only
            pairs[1, j] = [e, b16(30.0)]                            # bg only; fg high enough to be selected
            rows[0, j] = [e, b16(0.1), e, e]
            rows[1, j] = [b16(-0.2), e, e, b16(0.3)]
    _levels(conf, B, False, lg, bb)


# ------------------------------------------------------------------ DetectionLayer
def _detection(conf, win_px, image_shape, props, probs_bits, bbox_bits, pairs=PAIRS):
    """DetectionLayer on every dtype pair against the oracle on the widened arrays and the fp32 call."""
    from objectdetection_b200 import DetectionLayer
    probs, bbox = widen(probs_bits), widen(bbox_bits)
    B = props.shape[0]
    win = oracle.norm_boxes(win_px, image_shape[:2])
    want, wd = oracle.detection_forward(props, probs, bbox, win, conf.BBOX_STD_DEV, conf.DETECTION_MIN_THRESHOLD,
                                        conf.DETECTION_NMS_THRESHOLD, conf.DETECTION_POST_NMS_INSTANCES, debug=True)
    R = DetectionLayer(conf, image_shape, B, win_px, cu(props), cu(probs), cu(bbox), DEBUG=True)
    assert_bits(host(R.get_detections()), want, "fp32 call vs oracle")
    names = ("class_ids", "class_scores", "bbox_delta", "refined_proposals", "clipped_proposals", "keep_mask",
             "nms_keep_mask")
    for (pd, bd), pid in zip(pairs, IDS):
        D = DetectionLayer(conf, image_shape, B, win_px, cu(props), dev(probs_bits, pd), dev(bbox_bits, bd), DEBUG=True)
        assert_bits(host(D.get_detections()), want, f"{pid}: detections vs oracle")
        assert np.array_equal(host(D.class_ids), wd["class_ids"]), pid
        assert_bits(host(D.class_scores), wd["class_scores"], f"{pid}: class_scores vs oracle")
        assert_bits(host(D.clipped_proposals), wd["clipped_proposals"], f"{pid}: clipped vs oracle")
        assert np.array_equal(host(D.keep_mask), wd["keep_mask"]) and np.array_equal(host(D.nms_keep_mask), wd["nms_keep_mask"])
        same(D.get_detections(), R.get_detections(), f"{pid}: detections vs fp32 call")
        for n in names:
            same(getattr(D, n), getattr(R, n), f"{pid}: {n} vs fp32 call")
    return want


@gpu
def test_detection_debug_recipe_bf16(_cuda):
    """detection.py:285-310: seed 863, (1,8,4) / (1,8,4) / (1,8,4,4), window [131,0,893,1024]."""
    np.random.seed(863)
    props = np.array(np.random.random((1, 8, 4)), dtype="float32")
    probs = to_bits(np.random.random((1, 8, 4)))
    bbox = to_bits(np.random.random((1, 8, 4, 4)))
    _detection(Conf(), np.array([[131, 0, 893, 1024]], "int32"), [1024, 1024, 3], props, probs, bbox)


@gpu
def test_detection_coco_shape_bf16(_cuda):
    """BASELINE config 2: [2,1000,81] head outputs."""
    rs = np.random.RandomState(1234)
    props = _synth.rois_log_uniform(rs, 2, 1000)
    props[1, 900:] = 0
    probs, bbox = _synth.head_outputs(rs, 2, 1000, 81)
    win = np.array([[131, 0, 893, 1024], [0, 0, 1024, 1024]], "int32")
    det = _detection(Conf(), win, [1024, 1024, 3], props, to_bits(probs), to_bits(bbox))
    assert (det[:, :, 4] > 0).sum() > 50


@gpu
def test_detection_bf16_ties_nan_and_shapes(_cuda):
    """bf16-quantised probabilities with argmax and score ties; NaN at class 0 and at a later class; C = 1 and 2;
    N > 4096 (the bitonic-sort branch)."""
    rs = np.random.RandomState(9)
    conf = Conf()
    conf.DETECTION_POST_NMS_INSTANCES = 40
    win = np.array([[100, 0, 900, 1024], [0, 0, 1024, 1024]], "int32")
    B, N, C = 2, 400, 6
    props = _synth.random_boxes(rs, B * N).reshape(B, N, 4)
    probs, bbox = _synth.head_outputs(rs, B, N, C, boosted=0.9)
    probs = (np.round(probs * 8) / 8).astype(f32)                  # argmax ties and score ties
    pb = to_bits(probs)
    pb[0, 3, 0] = 0x7FC0                                            # NaN at class 0 wins
    pb[0, 5, 2] = 0xFFA1                                            # NaN at a later class is never taken
    pb[1, 7, :] = 0x7F81
    det = _detection(conf, win, [1024, 1024, 3], props, pb, to_bits(bbox))
    assert np.all(np.diff(det[:, :, 5], axis=1) <= 0)
    for C, N in ((1, 300), (2, 300), (2, 5000)):
        props = _synth.random_boxes(rs, B * N).reshape(B, N, 4)
        probs, bbox = _synth.head_outputs(rs, B, N, max(C, 2), boosted=0.5)
        _detection(conf, win, [1024, 1024, 3], props, to_bits(probs[..., :C]), to_bits(bbox[:, :, :C]))


# ------------------------------------------------------------------ losses
def _rpn_losses(tc, lg_bits, tb, pb_bits, pairs=PAIRS):
    """Loss.rpn_losses on every dtype pair: exact against the fp32 call, rtol 1e-6 against the oracle, pred_box_pos
    exact against both."""
    from objectdetection_b200.loss_optimize import Loss
    lg, pb = widen(lg_bits), widen(pb_bits)
    w = oracle.rpn_losses(tc, lg, tb, pb)
    r = Loss.rpn_losses(cu(tc), cu(lg), cu(tb), cu(pb), want_pos=True)
    for (ld, bd), pid in zip(pairs, IDS):
        g = Loss.rpn_losses(cu(tc), dev(lg_bits, ld), cu(tb), dev(pb_bits, bd), want_pos=True)
        for k in (0, 1):
            same(g[k], r[k], f"{pid}: loss {k} vs fp32 call")
            assert np.isclose(host(g[k]), w[k], rtol=1e-6, equal_nan=True), (pid, k, host(g[k]), w[k])
        same(g[2], r[2], f"{pid}: pred_box_pos vs fp32 call")
        assert_bits(host(g[2]), w[2][:g[2].shape[0]], f"{pid}: pred_box_pos vs oracle")
        pos, box = Loss.rpn_box_loss(cu(tb), dev(pb_bits, bd), cu(tc), tc.shape[0])
        same(box, r[1], f"{pid}: rpn_box_loss")
        same(pos, r[2], f"{pid}: rpn_box_loss pred_box_pos")
    return w


def _mrcnn_losses(ids, lg_bits, act, tb, pb_bits, pairs=PAIRS):
    from objectdetection_b200.loss_optimize import Loss
    lg, pb = widen(lg_bits), widen(pb_bits)
    w_pa, w_c, w_b = oracle.mrcnn_losses(ids, lg, act, tb, pb)
    r = Loss.mrcnn_losses(cu(ids), cu(lg), cu(act), cu(tb), cu(pb))
    for (ld, bd), pid in zip(pairs, IDS):
        g = Loss.mrcnn_losses(cu(ids), dev(lg_bits, ld), cu(act), cu(tb), dev(pb_bits, bd))
        same(g[0], r[0], f"{pid}: pred_active vs fp32 call")
        assert np.array_equal(host(g[0]), w_pa), pid
        for k, wk in ((1, w_c), (2, w_b)):
            same(g[k], r[k], f"{pid}: loss {k} vs fp32 call")
            assert np.isclose(host(g[k]), wk, rtol=1e-6, equal_nan=True), (pid, k, host(g[k]), wk)
        same(Loss.mrcnn_box_loss(cu(tb), dev(pb_bits, bd), cu(ids), batch_size=ids.shape[0]), r[2], f"{pid}: box loss alone")
        pa, c = Loss.mrcnn_class_loss(cu(ids), dev(lg_bits, ld), cu(act))
        same(pa, r[0], f"{pid}: class loss alone, pred_active")
        same(c, r[1], f"{pid}: class loss alone")


@gpu
def test_head_losses_bf16(_cuda):
    """The inputs of test_gpu_parity.test_head_losses, at bf16 precision."""
    from objectdetection_b200.data_processor import PreprareTrainData
    rs = np.random.RandomState(4)
    conf = Conf()
    P = PreprareTrainData(conf)
    A, B = P.anchors.shape[0], 2
    anc = host(P.anchors)
    gt = np.zeros((B, 20, 4))
    for b in range(B):
        gt[b] = np.round(np.clip(anc[rs.choice(A, 20, replace=False)] + rs.normal(0, 3, (20, 4)), 0, 1024))
        bad = (gt[b, :, 2] <= gt[b, :, 0]) | (gt[b, :, 3] <= gt[b, :, 1])
        gt[b, bad] = [100, 100, 164, 164]
    pp = np.stack([rs.permutation(A) for _ in range(B)]).astype(np.int32)
    _, tcls, tbox = P.build_rpn_targets(gt, perm_pos=pp, perm_neg=pp)
    tcls, tbox = host(tcls).reshape(B, A, 1), host(tbox).astype(f32)
    w = _rpn_losses(tcls, to_bits(rs.normal(0, 2, (B, A, 2))), tbox, to_bits(rs.normal(0, 1.5, (B, A, 4))))
    assert w[0] > 0 and w[1] > 0 and w[2].shape[0] > 0
    for Bm, R, C in ((2, 32, 4), (8, 200, 81)):
        ids = np.zeros((Bm, R), np.int32)
        if C == 4:
            ids[0, 2], ids[0, 3], ids[1, 4] = 1, 2, 1
        else:
            ids[:, :66] = rs.randint(1, C, (Bm, 66))
        tb2 = rs.random_sample((Bm, R, 4)).astype(f32)
        pb2 = to_bits(rs.random_sample((Bm, R, C, 4)))
        pb2[0, 2, ids[0, 2]] = to_bits(np.array([0.0, 1.0, 0.5, 1e-9], f32))     # exercises the epsilon clip
        act = (rs.random_sample((Bm, C)) > 0.3).astype(f32)
        act[:, 0] = 1
        _mrcnn_losses(ids, to_bits(rs.normal(0, 2, (Bm, R, C))), act, tb2, pb2)


@gpu
def test_head_losses_bf16_chunk_tail_no_targets_and_non_finite(_cuda):
    """A not a multiple of the 1024-anchor chunk, T = 0, and non-finite logits and predictions."""
    rs = np.random.RandomState(21)
    A, T = 2500, 8
    tc = rs.choice([-1, 0, 1], size=(3, A), p=[.3, .6, .1]).astype(np.int32)
    tc[1][tc[1] == 1] = 0
    lg = to_bits(rs.normal(0, 2, (3, A, 2)))
    pb = to_bits(rs.normal(0, 1, (3, A, 4)))
    tb = rs.normal(0, 1, (3, T, 4)).astype(f32)
    _rpn_losses(tc, lg, tb, pb)
    _rpn_losses(tc, lg, np.zeros((3, 0, 4), f32), pb)                               # T = 0
    lg2, pb2 = lg.copy(), pb.copy()
    nz = np.argwhere(tc != 0)
    for k, e in enumerate(EDGE_BITS):
        b, i = nz[k * 7]
        lg2[b, i, k % 2] = e
        pb2[b, i, k % 4] = e
    _rpn_losses(tc, lg2, tb, pb2)
    ids = np.zeros((2, 50), np.int32)
    ids[:, :20] = rs.randint(1, 5, (2, 20))
    lg3 = to_bits(rs.normal(0, 2, (2, 50, 5)))
    pb3 = to_bits(rs.random_sample((2, 50, 5, 4)))
    lg3[0, 0, 0], lg3[0, 1, 3], lg3[1, 2, 1] = 0x7F80, 0xFFC0, 0x7F7F
    pb3[0, 0, ids[0, 0], 1], pb3[1, 3, ids[1, 3], 2] = 0x7FC0, 0x8001
    act = np.ones((2, 5), f32)
    _mrcnn_losses(ids, lg3, act, rs.random_sample((2, 50, 4)).astype(f32), pb3)


# ------------------------------------------------------------------ dispatch, no copy
def _dispatch_worker():
    """Traces the bf16 and the fp32 calls of the three layers and prints the kernel names as JSON."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    from objectdetection_b200 import DetectionLayer, Proposals, utils
    from objectdetection_b200.loss_optimize import Loss
    conf = ShapesConfig()
    rs = np.random.RandomState(3)
    B = 2
    lg, bb = _level_bits(rs, conf, B)
    shapes = utils.get_resnet_stage_shapes(conf, conf.IMAGE_SHAPE)
    spec = utils.anchor_spec(conf.IMAGE_SHAPE, conf.RPN_ANCHOR_SCALES, conf.RPN_ANCHOR_RATIOS, shapes,
                             conf.RESNET_STRIDES, conf.RPN_ANCHOR_STRIDE)
    A = sum(t.size for t in lg) // (2 * B)
    props = cu(_synth.rois_log_uniform(rs, B, 300))
    probs, bbox = _synth.head_outputs(rs, B, 300, 81)
    tc = cu(rs.choice([-1, 0, 1], size=(B, A), p=[.3, .6, .1]).astype(np.int32))
    tb = cu(rs.normal(0, 1, (B, 16, 4)).astype(f32))
    ids = cu(rs.randint(0, 81, (B, 300)).astype(np.int32))
    act = cu(np.ones((B, 81), f32))
    win = np.array([[0, 0, 128, 128]] * B, "int32")
    res = {}
    for dt in (BF16, F32):
        L = [dev(t, dt) for t in lg]
        D = [dev(t, dt) for t in bb]
        pr, bx = cu(probs).to(dt), cu(bbox).to(dt)
        rl, rp = cu(rs.normal(0, 2, (B, A, 2)).astype(f32)).to(dt), cu(rs.normal(0, 1, (B, A, 4)).astype(f32)).to(dt)
        ml, mb = cu(rs.normal(0, 2, (B, 300, 81)).astype(f32)).to(dt), cu(rs.random_sample((B, 300, 81, 4)).astype(f32)).to(dt)
        fg = cu(np.full((B, A, 2), 0.5, f32))
        mt = cu(np.zeros((B, 300, 4), f32))
        calls = {
            "levels": lambda: Proposals(conf, B, anchor_spec=spec).run_levels(L, D),
            "flat": lambda: Proposals(conf, B, anchor_spec=spec).run(fg, rp),
            "detection": lambda: DetectionLayer(Conf(), [128, 128, 3], B, win, props, pr, bx),
            "rpn_loss": lambda: Loss.rpn_losses(tc, rl, tb, rp),
            "mrcnn_loss": lambda: Loss.mrcnn_losses(ids, ml, act, mt, mb),
        }
        for name, call in calls.items():
            call()                                            # workspace and host constants outside the window
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA], acc_events=True) as prof:
                call()
                torch.cuda.synchronize()
            res[f"{name}/{'bf16' if dt == BF16 else 'f32'}"] = [
                e.name for e in prof.events() if e.device_type == DeviceType.CUDA and not e.name.startswith(("Memcpy", "Memset"))]
    json.dump(res, sys.stdout)


KERNELS = {"levels": ["rpn_level_scores_kernel", "proposal_decode_kernel"], "flat": ["proposal_decode_kernel"],
           "detection": ["det_prepare_kernel"], "rpn_loss": ["rpn_loss_class_kernel", "rpn_loss_box_kernel"],
           "mrcnn_loss": ["mrcnn_loss_kernel"]}


@gpu
def test_bf16_dispatch_and_no_copy(_cuda):
    """bf16 calls launch the bf16 overloads and no conversion or copy kernel; fp32 calls launch the fp32 kernels.
    Traced in a process of its own (see test_gpu_roi_align_bf16.py)."""
    flags = ["-s"] if sys.flags.no_user_site else []
    r = subprocess.run([sys.executable, *flags, os.path.abspath(__file__), "--dispatch"], cwd=ROOT, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    res = json.loads(r.stdout)
    for name, kernels in KERNELS.items():
        names = res[f"{name}/bf16"]
        assert names, f"{name}: the CUDA kernel trace is empty"
        assert_launched(names, must=[k + "<" for k in kernels], must_not=["at::native", "copy"])
        for k in kernels:
            assert all("__nv_bfloat16" in n for n in names if k in n), names
        names = res[f"{name}/f32"]
        assert names, f"{name}: the CUDA kernel trace is empty"
        must = [f"od::{k}(" if k != "proposal_decode_kernel" else "od::proposal_decode_kernel<" for k in kernels]
        assert_launched(names, must=must, must_not=["__nv_bfloat16"])
    assert_launched(res["detection/f32"], must=["od::det_prepare_kernel("])


# ------------------------------------------------------------------ Python selection
@gpu
def test_inputs_the_bf16_kernels_do_not_take_are_converted_as_before(_cuda):
    """Misaligned bf16 views, float16, level lists of mixed dtype and host bf16 tensors are converted to fp32 as before
    and give the bits of the fp32 call."""
    from objectdetection_b200 import DetectionLayer, Proposals
    from objectdetection_b200.loss_optimize import Loss
    conf = ShapesConfig()
    rs = np.random.RandomState(8)
    B = 2
    lg, bb = _level_bits(rs, conf, B)
    from objectdetection_b200 import utils
    shapes = utils.get_resnet_stage_shapes(conf, conf.IMAGE_SHAPE)
    spec = utils.anchor_spec(conf.IMAGE_SHAPE, conf.RPN_ANCHOR_SCALES, conf.RPN_ANCHOR_RATIOS, shapes,
                             conf.RESNET_STRIDES, conf.RPN_ANCHOR_STRIDE)

    def run(L, D):
        return Proposals(conf, B, anchor_spec=spec).run_levels(L, D)

    want = run([dev(t, F32) for t in lg], [dev(t, F32) for t in bb])

    def off2(bits):
        """A contiguous bf16 view 2 bytes past an aligned start."""
        flat = torch.zeros(bits.size + 1, dtype=BF16, device="cuda")
        flat[1:] = dev(bits, BF16).reshape(-1)
        v = flat[1:].view(bits.shape)
        assert v.data_ptr() % 4 == 2
        return v

    cases = {
        "misaligned deltas": ([dev(t, BF16) for t in lg], [off2(bb[0])] + [dev(t, BF16) for t in bb[1:]]),
        "misaligned logits": ([off2(lg[0])] + [dev(t, BF16) for t in lg[1:]], [dev(t, BF16) for t in bb]),
        "float16": ([dev(t, F32).half() for t in lg], [dev(t, F32).half() for t in bb]),
        "mixed logits": ([dev(lg[0], BF16)] + [dev(t, F32) for t in lg[1:]], [dev(t, BF16) for t in bb]),
        "mixed deltas": ([dev(t, BF16) for t in lg], [dev(t, F32) for t in bb[:-1]] + [dev(bb[-1], BF16)]),
        "host bf16": ([dev(t, BF16).cpu() for t in lg], [dev(t, BF16).cpu() for t in bb]),
    }
    for what, (L, D) in cases.items():
        if what == "float16":
            ref = run([t.float() for t in L], [t.float() for t in D])     # float16 values, as the fp32 call sees them
        else:
            ref = want
        same(run(L, D), ref, what)
    # DetectionLayer and the losses: misaligned, float16 and host bf16
    rs = np.random.RandomState(9)
    props = cu(_synth.rois_log_uniform(rs, B, 200))
    probs, bbox = _synth.head_outputs(rs, B, 200, 9)
    pbits, bbits = to_bits(probs), to_bits(bbox)
    win = np.array([[0, 0, 1024, 1024]] * B, "int32")

    def det(p, b):
        return DetectionLayer(Conf(), [1024, 1024, 3], B, win, props, p, b).get_detections()
    ref = det(dev(pbits, F32), dev(bbits, F32))
    flat = torch.zeros(bbits.size + 2, dtype=BF16, device="cuda")
    flat[2:] = dev(bbits, BF16).reshape(-1)
    mis = flat[2:].view(bbits.shape)
    assert mis.data_ptr() % 8 == 4
    same(det(dev(pbits, BF16), mis), ref, "detection: misaligned boxes")
    same(det(dev(pbits, BF16).cpu(), dev(bbits, BF16).cpu()), ref, "detection: host bf16")
    same(det(dev(pbits, F32).half(), dev(bbits, F32).half()), det(dev(pbits, F32).half().float(), dev(bbits, F32).half().float()),
         "detection: float16")
    A = 3000
    tc = rs.choice([-1, 0, 1], size=(B, A), p=[.3, .6, .1]).astype(np.int32)
    lbits, rbits = to_bits(rs.normal(0, 2, (B, A, 2))), to_bits(rs.normal(0, 1, (B, A, 4)))
    tb = cu(rs.normal(0, 1, (B, 32, 4)).astype(f32))
    r = Loss.rpn_losses(cu(tc), dev(lbits, F32), tb, dev(rbits, F32), want_pos=True)
    flat = torch.zeros(rbits.size + 2, dtype=BF16, device="cuda")
    flat[2:] = dev(rbits, BF16).reshape(-1)
    for what, (lt, pt) in {"misaligned pred": (dev(lbits, BF16), flat[2:].view(rbits.shape)),
                           "host bf16": (dev(lbits, BF16).cpu(), dev(rbits, BF16).cpu())}.items():
        g = Loss.rpn_losses(cu(tc), lt, tb, pt, want_pos=True)
        for k in range(3):
            same(g[k], r[k], f"rpn losses, {what}: {k}")


if __name__ == "__main__" and sys.argv[1:] == ["--dispatch"]:
    _dispatch_worker()
