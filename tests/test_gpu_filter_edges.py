"""GPU parity at the input values where the kernels' cheap pre-filters could decide differently from the exact
arithmetic behind them: very tall Faster R-CNN images with near-threshold pairs of tiny boxes, NMS boxes made of signed
zeros, one-ulp overlaps, subnormals, infinities and NaNs, RPN-target boxes closer together than fp32 can resolve,
top-k rows full of infinities, NaNs and subnormals, and decoders fed deltas that overflow exp. Every result is compared
with the CPU oracle bit for bit (NaN equal to NaN), integer outputs exactly. The box sets come from the numpy replays of
test_filter_replays.py."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import _synth  # noqa: E402
import test_filter_replays as replays  # noqa: E402
from test_gpu_parity import _check_detection, _check_proposals, assert_bits, cu, host  # noqa: E402

import oracle  # noqa: E402
from objectdetection_b200.config import ShapesConfig, config as Conf  # noqa: E402

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu
f32 = np.float32


@pytest.fixture(scope="module", autouse=True)
def _need_cuda():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (there is no CPU path)")


def _bits(x):
    return np.asarray(x, f32).view(np.uint32)


# ------------------------------------------------------------------ Faster R-CNN: fp32 screen vs image size
def _frcnn_pair_inputs(rs, image_h, image_w, thr, adversarial, fh=112, fw=3, tries=256):
    """RPN outputs [1,fh,fw,18] / [1,fh,fw,36] (fp64) whose decoded, clipped boxes are isolated pairs of 1-4 px boxes
    with IoU near thr, in columns 12 px apart and rows 10 px apart at the bottom of the image. Pair s is anchors 2s
    (higher score) and 2s + 1. With `adversarial`, each pair is the first of `tries` random candidates that the fp32
    screen misjudges for every quotient __fdividef may return, when one exists. Returns (probs, bbox, #misjudged)."""
    base = oracle.FRCNN_BASE_ANCHORS
    na = base.shape[0]
    total = fh * fw * na
    S = total // 2
    pos = np.arange(total) // na
    anchors = base[np.arange(total) % na] + np.stack([(pos % fw) * 16, (pos // fw) * 16] * 2, 1)
    cols = (image_w - 4) // 12
    slot_x = 2.0 + 12.0 * (np.arange(S) % cols)
    slot_y = image_h - 14.0 - 10.0 * (np.arange(S) // cols)
    assert slot_y.min() > 0

    def deltas_for(box, anc):   # inverse of corner_pixels_to_center_inv (proposals.py:286-309), fp64
        aw, ah = anc[..., 2] - anc[..., 0] + 1, anc[..., 3] - anc[..., 1] + 1
        acx, acy = anc[..., 0] + aw / 2, anc[..., 1] + ah / 2
        pw, ph = box[..., 2] - box[..., 0], box[..., 3] - box[..., 1]
        cx, cy = (box[..., 0] + box[..., 2]) / 2, (box[..., 1] + box[..., 3]) / 2
        with np.errstate(divide="ignore"):   # a 1 px side is pw = 0: dw = -inf, exp(-inf) = 0
            return np.stack([(cx - acx) / aw, (cy - acy) / ah, np.log(pw / aw), np.log(ph / ah)], -1)

    def decoded(d, anc):
        b = oracle.frcnn_decode(anc.reshape(-1, 4), d.reshape(-1, 4)).reshape(d.shape)
        b[..., 0::2] = np.clip(b[..., 0::2], 0, image_w - 1)
        b[..., 1::2] = np.clip(b[..., 1::2], 0, image_h - 1)
        return b

    # candidate pairs with corners in [0, 1) (boxes within 6 px of it), moved to each slot
    bi, bj = replays.near_threshold_pairs(rs, S * tries, thr, 0.0, 13.0)
    shift = np.stack([slot_x, slot_y] * 2, 1).repeat(tries, 0)
    bi, bj = bi + shift, bj + shift
    a_i, a_j = anchors[0::2][:S].repeat(tries, 0), anchors[1::2][:S].repeat(tries, 0)
    d_i, d_j = deltas_for(bi, a_i), deltas_for(bj, a_j)
    di, dj = decoded(d_i, a_i), decoded(d_j, a_j)
    hit, miss = replays.frcnn_screen(di, dj, thr, certain=True)
    exact = replays.frcnn_exact(di, dj, thr)
    wrong = ((hit & ~exact) | (miss & exact)).reshape(S, tries)
    pick = np.argmax(wrong, 1) if adversarial else np.zeros(S, int)
    rows = np.arange(S) * tries + pick
    d = np.zeros((total, 4))
    d[0:2 * S:2], d[1:2 * S:2] = d_i[rows], d_j[rows]
    score = np.zeros(total)
    score[:2 * S] = 1.0 - np.arange(2 * S) / (2.0 * S)          # pair order = visiting order
    probs = np.zeros((1, fh, fw, 2 * na))
    probs[0, ..., :na] = score.reshape(fh, fw, na)
    bbox = d.reshape(1, fh, fw, 4 * na)
    return probs, bbox, int(wrong[np.arange(S), pick].sum())


@pytest.mark.parametrize("image_h", [8192, 131072])
def test_frcnn_tall_image_near_threshold_pairs(image_h):
    """8192 x 48 keeps the fp32 screen; 131072 x 48 is past its bound, where the screen alone would misjudge the
    pairs chosen here (the parent of the bound check failed this case). Both must equal the fp64 reference."""
    from objectdetection_b200 import fasterrcnn
    rs = np.random.RandomState(image_h % 1000)
    probs, bbox, misjudged = _frcnn_pair_inputs(rs, image_h, 48, 0.7, adversarial=image_h > 8192)
    if image_h > 8192:
        assert misjudged > 100, misjudged
    n = probs.shape[1] * probs.shape[2] * 9
    P = fasterrcnn.Proposals('test', probs, bbox, image_shape=(image_h, 48, 3), nms_threshold=0.7, pre_nms_top_n=n,
                             post_nms_top_n=n, min_box_hw=1)
    got = host(P.get_proposals())
    want = oracle.frcnn_proposals(probs, bbox, image_h, 48, n, n, 0.7, min_hw=1)
    S = n // 2
    assert S < want.shape[0] < n                  # every pair keeps its first box; some second boxes survive
    assert got.shape == want.shape, (got.shape, want.shape)
    assert np.array_equal(_bits(got), _bits(want))


def test_frcnn_refuses_empty_image_size():
    from objectdetection_b200 import fasterrcnn
    rs = np.random.RandomState(0)
    probs, bbox = rs.random_sample((1, 4, 4, 18)), rs.normal(0, 0.5, (1, 4, 4, 36))
    for shape in ((0, 48, 3), (48, 0, 3), (-5, 48, 3)):
        with pytest.raises(ValueError):
            fasterrcnn.Proposals('test', probs, bbox, image_shape=shape)


# ------------------------------------------------------------------ NMS on the adversarial box set
@pytest.mark.parametrize("thr", [0.0, 1e-7, 0.5, 1.0])
def test_nms_adversarial_boxes(thr):
    """The CPU replay's box set (signed zeros, shared edges, one-ulp overlaps, subnormal sides, infinities, NaN in
    every position, flipped and overflowing boxes) through non_max_suppression, three images: as built, shuffled with
    tied, signed-zero and NaN scores, and with ragged num_valid."""
    from objectdetection_b200.proposals import non_max_suppression
    rs = np.random.RandomState(int(thr * 10) + 1)
    boxes = replays.nms_adversarial_boxes(rs)
    K = boxes.shape[0]
    b3 = np.stack([boxes, boxes[rs.permutation(K)], boxes])
    s3 = rs.random_sample((3, K)).astype(f32)
    s3[1] = np.round(s3[1] * 8) / 8
    s3[1, :6] = [-0.0, 0.0, np.nan, -np.nan, np.inf, -np.inf]
    s3[1, 6:8] = np.array([0xFFC00000, 0x7FC01234], np.uint32).view(f32)
    nv = np.array([K, K, K - 37], np.int32)
    for max_out in (K, 7):
        keep, num = non_max_suppression(cu(b3), cu(s3), max_out, thr, num_valid=nv)
        keep, num = host(keep), host(num)
        for b in range(3):
            want = oracle.nms(b3[b, :nv[b]], s3[b, :nv[b]], max_out, thr)
            assert num[b] == want.shape[0], (b, max_out, num[b], want.shape[0])
            assert np.array_equal(keep[b, :num[b]], want) and np.all(keep[b, num[b]:] == -1), (b, max_out)


# ------------------------------------------------------------------ RPN targets: boxes below fp32 resolution
@pytest.mark.parametrize("m", [1e3, 2.0 ** 24, 1e7])
def test_rpn_targets_near_resolution_boxes(m):
    """Anchors and GT boxes whose fp64 edges are closer than fp32 resolves at magnitude m (slivers of overlap, touching
    edges, zero-width GT): a missed sliver would zero a GT's only positive IoU and move its best anchor. Fused (G <= 256)
    and per-GT (G padded past 256) kernels, against the fp64 numpy oracle."""
    from objectdetection_b200.data_processor import PreprareTrainData
    rs = np.random.RandomState(7)
    anchors, gts = replays.rpn_near_resolution_boxes(rs, m)
    P = PreprareTrainData(ShapesConfig())
    P.anchors = cu(anchors)
    P.anchor_area = (P.anchors[:, 2] - P.anchors[:, 0]) * (P.anchors[:, 3] - P.anchors[:, 1])
    A, G, T = anchors.shape[0], gts.shape[0], P.max_rpn_targets
    assert G <= 256
    pp = np.stack([rs.permutation(A) for _ in range(2)]).astype(np.int32)
    pn = np.stack([rs.permutation(A) for _ in range(2)]).astype(np.int32)
    w_pos, w_cls, w_bbox, w_counts = oracle.rpn_targets(anchors, gts, pp[0], pn[0], T, P.bbox_std_dev)
    assert w_counts[2] > 0
    for pad in (G, 300):
        gt = np.zeros((2, pad, 4))
        gt[:, :G] = gts
        pos, cls, bbox, counts = P.build_rpn_targets(gt, perm_pos=pp[[0, 0]], perm_neg=pn[[0, 0]],
                                                     gt_count=np.array([G, G], np.int32), return_counts=True)
        pos, cls, bbox, counts = host(pos), host(cls), host(bbox), host(counts)
        for b in range(2):
            assert np.array_equal(counts[b], w_counts), (pad, counts[b], w_counts)
            assert np.array_equal(cls[b], w_cls), pad
            n = w_counts[2]
            assert np.array_equal(pos[b, :n], w_pos) and not pos[b, n:].any()
            with np.errstate(invalid="ignore"):
                assert np.allclose(bbox[b], w_bbox, rtol=1e-13, atol=0, equal_nan=True)


# ------------------------------------------------------------------ top-k over non-finite scores
def _special_row(rs, cols, n_nan, n_pinf):
    """N(0,1) scores with n_nan NaNs (both signs, several payloads), n_pinf +inf, and -inf, subnormals and +-0."""
    row = rs.normal(0, 1, cols).astype(f32)
    nans = np.array([0x7FC00000, 0xFFC00000, 0x7FC01234, 0xFFFFFFFF, 0x7F800001], np.uint32).view(f32)
    idx = rs.permutation(cols)
    row[idx[:n_nan]] = nans[rs.randint(0, nans.size, n_nan)]
    row[idx[n_nan:n_nan + n_pinf]] = np.inf
    rest = idx[n_nan + n_pinf:]
    row[rest[:50]] = -np.inf
    row[rest[50:100]] = np.array([1, 2, 0x007FFFFF, 0x80000001, 0x80000000, 0], np.uint32).view(f32)[rs.randint(0, 6, 50)]
    return row


@pytest.mark.parametrize("cols,k,n_nan,n_pinf", [
    (5000, 300, 100, 100),          # mixed row: k ends among the finite scores
    (5000, 5000, 2500, 500),        # take-all
    (100000, 1000, 40000, 10),      # k ends inside the NaN bucket; 40000 candidates > the 16384-entry buffer
    (100000, 8000, 5000, 40000),    # k ends inside the +inf bucket; 40000 candidates > the 32768-entry buffer
    (70000, 20000, 0, 0),           # k > 16384 (global sort) with -inf, subnormals and +-0 ties
])
def test_topk_non_finite_scores(cols, k, n_nan, n_pinf):
    """Indices and value bits against oracle.topk: every NaN is one value above +inf, -0 ties +0, ties -> lower index.
    The last row of every batch is all NaN (mixed signs and payloads)."""
    from objectdetection_b200.proposals import top_k
    rs = np.random.RandomState(cols + k)
    s = np.stack([_special_row(rs, cols, n_nan, n_pinf) for _ in range(2)] + [_special_row(rs, cols, cols - 100, 0)])
    v, i = top_k(cu(s), k)
    wv, wi = oracle.topk(s, k)
    assert np.array_equal(host(i), wi)
    assert np.array_equal(_bits(host(v)), _bits(wv))


# ------------------------------------------------------------------ decoders: overflowing deltas, NaN scores
def test_proposals_overflowing_deltas_and_nan_scores():
    """ProposalLayer (DEBUG) with deltas up to +-1e3 (exp overflows: decoded boxes inf or NaN) and NaN foreground
    scores of both signs: every intermediate against the oracle."""
    from objectdetection_b200 import Proposals, utils
    conf = ShapesConfig()
    rs = np.random.RandomState(11)
    shapes = utils.get_resnet_stage_shapes(conf, conf.IMAGE_SHAPE)
    anchors = oracle.gen_anchors(conf.IMAGE_SHAPE, 2, conf.RPN_ANCHOR_SCALES, conf.RPN_ANCHOR_RATIOS, shapes,
                                 conf.RESNET_STRIDES, 1)
    A = anchors.shape[1]
    probs, bbox = _synth.rpn_outputs(rs, 2, A)
    big = rs.random_sample((2, A)) < 0.3
    bbox[big] = np.clip(rs.normal(0, 400, (int(big.sum()), 4)), -1e3, 1e3).astype(f32)
    bbox[0, :8] = [[1e3, 1e3, 1e3, 1e3], [-1e3, -1e3, -1e3, -1e3], [0, 0, 1e3, -1e3], [0, 0, -1e3, 1e3],
                   [1e3, -1e3, 0, 0], [0, 0, 500, 0], [np.nan, 0, 0, 0], [0, 0, np.inf, 0]]
    nan_rows = rs.random_sample((2, A)) < 0.02
    probs[..., 1][nan_rows] = np.array([0x7FC00000, 0xFFC00000], np.uint32).view(f32)[rs.randint(0, 2, int(nan_rows.sum()))]
    P = Proposals(conf, 2, cu(probs), cu(bbox), cu(anchors), DEBUG=True)
    want = _check_proposals(P, probs, bbox, anchors, conf)
    assert np.isnan(want).any()                                 # NaN boxes survive clip and NMS
    assert_bits(host(Proposals(conf, 2, cu(probs), cu(bbox), cu(anchors)).get_proposals()), want, "proposals")
    _, dbg = oracle.proposal_forward(probs, bbox, anchors, conf.RPN_BBOX_STDDEV, conf.PRE_NMS_ROIS_COUNT,
                                     conf.POST_NMS_ROIS_INFERENCE, conf.RPN_NMS_THRESHOLD, debug=True)
    assert not np.isfinite(dbg["anchor_delta"]).all()          # the overflow reached the decoded boxes
    assert np.isnan(dbg["scores"]).any()                        # NaN scores were among the top-K
    assert want.shape == (2, conf.POST_NMS_ROIS_INFERENCE, 4)


def test_detection_nan_probabilities_and_overflowing_deltas():
    """DetectionLayer (DEBUG) with all-NaN and partly NaN class-probability rows and deltas up to +-1e3."""
    rs = np.random.RandomState(12)
    B, N, C = 2, 600, 81
    props = _synth.rois_log_uniform(rs, B, N)
    probs, bbox = _synth.head_outputs(rs, B, N, C, boosted=0.5)
    probs[0, :20] = np.nan
    probs[1, :20] = np.array([0xFFC00000], np.uint32).view(f32)[0]
    part = rs.random_sample((B, N, C)) < 0.01
    probs[part] = np.nan
    big = rs.random_sample((B, N, C)) < 0.2
    bbox[big] = np.clip(rs.normal(0, 400, (int(big.sum()), 4)), -1e3, 1e3).astype(f32)
    bbox[:, 20:40] = 1e3
    bbox[:, 40:60] = -1e3
    win = np.array([[131, 0, 893, 1024], [0, 0, 1024, 1024]], "int32")
    det = _check_detection(Conf(), win, [1024, 1024, 3], props, probs, bbox)
    assert (det[:, :, 4] > 0).sum() > 20
