"""The float64 references of tests/_f64_refs.py on answers worked out by hand and against torch float64, then the
oracle against them on the inputs of tests/test_gpu_unpinned_outputs.py. No GPU: this pins the oracle's mask targets
and head losses to something other than the kernels they are compared with."""
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import _f64_refs as ref  # noqa: E402

import oracle  # noqa: E402
from objectdetection_b200.config import config as Conf  # noqa: E402
import test_gpu_unpinned_outputs as cases  # noqa: E402

torch = pytest.importorskip("torch")
F = torch.nn.functional
f32 = np.float32


# ------------------------------------------------------------------ mask targets: known answers
def test_mask_exact_tie_rounds_half_to_even():
    """Mw = 3, mw = 5, box [0,0,1,1]: the taps land on x = 0, 0.5, 1, 1.5, 2 of the columns [0,1,0], so the values
    are 0, 0.5, 1, 0.5, 0; exact in fp32, hence decidable, and tf.round sends 0.5 to 0."""
    masks = np.zeros((3, 3, 1), f32)
    masks[:, 1, 0] = 1
    for mini in (True, False):
        v, dec = ref.mask_targets_f64(np.array([[0, 0, 1, 1]], f32), np.array([[0, 0, 1, 1]], f32), [0], masks, (3, 5),
                                      mini)
        assert np.array_equal(v[0], np.tile([0, 0.5, 1, 0.5, 0], (3, 1))) and dec.all()
        assert np.array_equal(np.round(v[0]), np.tile([0, 0, 1, 0, 0], (3, 1)))
    # a tie reached through inexact arithmetic is not decidable: columns [0, 0.75, 0], 7 taps, x = 2/3 gives 0.5
    masks[:, 1, 0] = 0.75
    v, dec = ref.mask_targets_f64(np.array([[0, 0, 1, 1]], f32), np.zeros((1, 4), f32), [0], masks, (3, 7), False)
    assert abs(v[0, 0, 2] - 0.5) < 1e-12 and not dec[0, :, 2].any() and dec[0, :, 3].all()


def test_mask_size_one_uses_the_centre():
    """A mask size of 1 samples the box centre, 0.5 (y1 + y2) (M - 1): box y 0.2..0.6, x 0.4..0.8 over a 5x5 ramp
    v = (4 y + x) / 24 gives y = 1.6, x = 2.4, v = 8.8 / 24."""
    yy, xx = np.mgrid[0:5, 0:5]
    masks = ((4 * yy + xx) / 24.0).astype(f32)[..., None]
    v, dec = ref.mask_targets_f64(np.array([[0.2, 0.4, 0.6, 0.8]]), np.zeros((1, 4)), [0], masks, (1, 1), False)
    assert v.shape == (1, 1, 1) and abs(v[0, 0, 0] - 8.8 / 24) < 1e-7 and dec.all()
    v, _ = ref.mask_targets_f64(np.array([[0.2, 0.4, 0.6, 0.8]]), np.zeros((1, 4)), [0], masks, (1, 3), False)
    assert np.allclose(v[0, 0], [(4 * 1.6 + 1.6) / 24, 8.8 / 24, (4 * 1.6 + 3.2) / 24])


def test_mask_degenerate_gt_and_outside_rois():
    """gt_h = 0 or gt_w = 0 with mini masks: the box in the GT frame is infinite or NaN, every sample falls outside,
    the target is all zero and decidable. A full-mask ROI reaching above the mask: the rows outside extrapolate to 0."""
    masks = np.ones((4, 4, 2), f32)
    gt = np.array([[0.3, 0.2, 0.3, 0.7], [0.2, 0.4, 0.8, 0.4]], f32)
    rois = np.array([[0.25, 0.2, 0.35, 0.7], [0.3, 0.2, 0.4, 0.7], [0.2, 0.3, 0.8, 0.5]], f32)
    v, dec = ref.mask_targets_f64(rois, gt, [0, 0, 1], masks, (7, 7), True)
    assert not v.any() and dec.all()
    masks = np.ones((3, 3, 1), f32)
    v, dec = ref.mask_targets_f64(np.array([[-1, 0, 1, 1]], f32), np.zeros((1, 4)), [0], masks, (3, 3), False)
    assert np.array_equal(v[0], [[0, 0, 0], [1, 1, 1], [1, 1, 1]]) and dec.all()    # rows at y = -2, 0, 2


def test_gt_assignment_maps_compacted_to_original_rows():
    """Class-0 rows before and between the valid GT boxes: the compacted index and the original row differ."""
    gt = np.array([[0, 0, 1, 1], [0.1, 0.1, 0.5, 0.5], [0, 0, 1, 1], [0.5, 0.5, 0.9, 0.9], [0.5, 0.5, 0.9, 0.9]], f32)
    cls = np.array([0, 4, 0, 7, 9], np.int32)
    rois = np.array([[0.5, 0.5, 0.9, 0.85], [0.1, 0.1, 0.5, 0.45]], f32)
    rows, comp, amb = ref.gt_assignment_f64(rois, gt, cls)
    assert rows.tolist() == [3, 1] and comp.tolist() == [1, 0] and amb.tolist() == [True, False]


# ------------------------------------------------------------------ losses: known answers
def test_cross_entropy_known_answers():
    """Two-class CE by hand: log(e^1 + e^3) - 1 = 2 + log1p(e^-2); equal logits log 2; -inf on the other side 0;
    targets 2 and -7 count as background (label equal(., 1)), 0 is left out."""
    tc = np.array([[1, -1, 0, 2, -7, 1]], np.int32)
    lg = np.array([[[0, 0], [1, 3], [50, -50], [3, 1], [0, 0], [-np.inf, 2]]], f32)
    ce = [np.log(2), 2 + np.log1p(np.exp(-2)), np.log1p(np.exp(-2)), np.log(2), 0.0]
    cl, cb, bl, bb, pos = ref.rpn_losses_f64(tc, lg, np.zeros((1, 0, 4), f32), np.zeros((1, 6, 4), f32))
    assert abs(cl - np.mean(ce)) < 1e-15 and 0 < cb < 1e-5 and bl == 0 and pos.shape == (2, 4)
    # a gap beyond the fp32 range is +inf there; a +inf or NaN logit is NaN
    for row, want in (([3e38, -3e38], np.inf), ([np.inf, 0], np.nan), ([1.0, np.nan], np.nan)):
        cl = ref.rpn_losses_f64(np.array([[1]]), np.array([[row]], f32), np.zeros((1, 0, 4)), np.zeros((1, 1, 4)))[0]
        assert cl == want or (np.isnan(cl) and np.isnan(want)), (row, cl)


def test_smooth_l1_known_answers():
    """0.5 d^2 below 1, d - 0.5 from 1 on: d = 0.5 -> 0.125, 1 -> 0.5, nextafter(1, 0) -> 0.5 (1 - 2^-24)^2,
    2 -> 1.5; d = 2e19 squares past the fp32 range and the element is NaN."""
    below = float(np.nextafter(f32(1), f32(0)))
    l, _ = ref.smooth_l1_f64(np.zeros(5), [0.5, -1, below, 2, 2e19])
    assert l[:4].tolist() == [0.125, 0.5, 0.5 * below * below, 1.5] and np.isnan(l[4])
    l, _ = ref.smooth_l1_f64([1e19], [-1e19])
    assert np.isnan(l[0])


def test_bce_known_answers():
    """-(t log o + (1 - t) log(1 - o)) with o clipped to [eps, 1 - eps] in fp32: p = 0.5 -> log 2 for any t,
    p = 0.2, t = 0.5 -> -(0.5 log 0.2 + 0.5 log 0.8), p = 1, t = 1 -> -log(1 - eps), p <= 0 -> o = eps."""
    eps, hi = float(f32(1e-7)), float(f32(1) - f32(1e-7))
    t = np.array([1, 0.3, 0.5, 1, 0, 0, 1.5])
    p = np.array([0.5, 0.5, 0.2, 1, 0, -3, 2])
    want = -(t * np.log(np.clip(p, eps, hi)) + (1 - t) * np.log(1 - np.clip(p, eps, hi)))
    l, _ = ref.bce_f64(t, p)
    assert np.allclose(l, want, rtol=1e-9, atol=1e-15)
    assert abs(l[0] - np.log(2)) < 1e-15 and abs(l[3] + np.log(hi)) < 1e-15 and abs(l[4] + np.log1p(-eps)) < 1e-15
    assert hi == 1 - 2 ** -23                                                           # the fp32 1 - eps, not 1
    assert np.isnan(ref.bce_f64([1], [np.nan])[0][0])


def test_first_max_and_inactive_classes():
    """The strict '>' scan: the first of equal maxima, a NaN at index 0 stays, a later NaN never wins; no active
    predicted class gives 0/0 = NaN."""
    x = np.array([[1, 3, 3, 2], [np.nan, 5, 1, 0], [0, np.nan, 4, 4], [-np.inf] * 4], f32)
    arg, m = ref.first_max(x)
    assert arg.tolist() == [1, 0, 2, 0] and np.isnan(m[1]) and m[2] == 4
    ids = np.zeros((1, 2), np.int32)
    lg = np.array([[[1, 2], [3, 0]]], f32)
    pa, cl, _, bl, _ = ref.mrcnn_losses_f64(ids, lg, np.array([[0, 0]], f32), np.zeros((1, 2, 4)), np.zeros((1, 2, 2, 4)))
    assert np.isnan(cl) and bl == 0 and not pa.any()
    pa, cl, _, _, _ = ref.mrcnn_losses_f64(ids, lg, np.array([[1, 0]], f32), np.zeros((1, 2, 4)), np.zeros((1, 2, 2, 4)))
    assert pa.tolist() == [[0, 1]] and abs(cl - np.log1p(np.exp(-3))) < 1e-15       # only row 1 (argmax 0) counts


def test_losses_match_torch_float64():
    """Second opinion on random inputs: torch float64 cross_entropy, smooth_l1_loss and binary_cross_entropy."""
    rs = np.random.RandomState(1)
    B, A, T = 3, 700, 20
    tc = rs.choice([-1, 0, 1], size=(B, A), p=[.3, .6, .1]).astype(np.int32)
    lg = rs.normal(0, 3, (B, A, 2)).astype(f32)
    tb, pb = rs.normal(0, 1, (B, T, 4)).astype(f32), rs.normal(0, 2, (B, A, 4)).astype(f32)
    cl, cb, bl, bb, _ = ref.rpn_losses_f64(tc, lg, tb, pb)
    sel = torch.from_numpy(tc != 0)
    want = F.cross_entropy(torch.from_numpy(lg).double()[sel], torch.from_numpy(tc == 1)[sel].long())
    assert abs(cl - float(want)) < 1e-12
    pr = np.concatenate([pb[b][tc[b] == 1][:T] for b in range(B)])
    tg = np.concatenate([tb[b, :min(int((tc[b] == 1).sum()), T)] for b in range(B)])
    assert abs(bl - float(F.smooth_l1_loss(torch.from_numpy(pr).double(), torch.from_numpy(tg).double()))) < 1e-12
    R, C = 300, 81
    ids = np.where(rs.random_sample((B, R)) < 0.5, 0, rs.randint(1, C, (B, R))).astype(np.int32)
    lg2 = rs.normal(0, 3, (B, R, C)).astype(f32)
    act = (rs.random_sample((B, C)) > 0.3).astype(f32)
    tb2, pb2 = rs.random_sample((B, R, 4)).astype(f32), rs.uniform(0.01, 0.99, (B, R, C, 4)).astype(f32)
    pa, cl2, _, bl2, _ = ref.mrcnn_losses_f64(ids, lg2, act, tb2, pb2)
    ce = F.cross_entropy(torch.from_numpy(lg2).double().reshape(-1, C), torch.from_numpy(ids).long().reshape(-1),
                         reduction="none")
    w = torch.from_numpy(act[0]).double()[torch.from_numpy(lg2).reshape(-1, C).argmax(-1)]
    assert np.array_equal(pa.reshape(-1), w.numpy()) and abs(cl2 - float((ce * w).sum() / w.sum())) < 1e-12
    m = ids > 0
    want = F.binary_cross_entropy(torch.from_numpy(pb2[m, ids[m]]).double(), torch.from_numpy(tb2[m]).double())
    assert abs(bl2 - float(want)) < 1e-12


# ------------------------------------------------------------------ the oracle against the references
CPU_MASK_CASES = [c for c in cases.MASK_CASES if c != "full_image_1024"]


@pytest.mark.parametrize("mini", [True, False])
@pytest.mark.parametrize("case", CPU_MASK_CASES)
def test_oracle_mask_targets_vs_f64(case, mini):
    shape, R, props, cls, gt, pp, pn, masks = cases.mask_case(case)
    B = props.shape[0]
    rois = np.zeros((B, R, 4), f32)
    targets = np.zeros((B, R) + shape, f32)
    n_pos, assign = np.zeros(B, int), np.zeros((B, R), np.int32)
    for b in range(B):
        rois[b], _, _, wd = oracle.detection_targets(props[b], cls[b], gt[b], pp[b], pn[b], R, Conf.BBOX_STD_DEV)
        targets[b] = oracle.mask_targets(rois[b], cls[b], gt[b], masks[b], wd, shape, mini)
        n_pos[b], assign[b] = wd["counts"][4], wd["gt_assignment"]
    cases.check_masks_against_f64(shape, mini, props, cls, gt, masks, rois, n_pos, assign, targets)
    if case.startswith("pad_"):
        moved = [not np.array_equal(np.nonzero(cls[b])[0], np.arange(np.count_nonzero(cls[b]))) for b in range(B)]
        assert all(moved), "the case must move GT rows away from their compacted index"


@pytest.mark.parametrize("A,B", [s for s in cases.RPN_SHAPES if s[0] * s[1] < 10 ** 6])
def test_oracle_rpn_losses_vs_f64(A, B):
    tc, lg, tb, pb = cases.rpn_case(A, B)
    cl, cb, bl, bb, pos = ref.rpn_losses_f64(tc, lg, tb, pb)
    o_cl, o_bl, o_pos = oracle.rpn_losses(tc, lg, tb, pb)
    ref.assert_loss(o_cl, cl, cb, "class")
    ref.assert_loss(o_bl, bl, bb, "box")
    assert np.array_equal(o_pos, pos)


def test_oracle_rpn_losses_non_finite_vs_f64():
    for name, tc, lg, tb, pb in cases.rpn_nonfinite_cases():
        cl, cb, bl, bb, _ = ref.rpn_losses_f64(tc, lg, tb, pb)
        o_cl, o_bl, _ = oracle.rpn_losses(tc, lg, tb, pb)
        ref.assert_loss(o_cl, cl, cb, f"{name} class")
        ref.assert_loss(o_bl, bl, bb, f"{name} box")


@pytest.mark.parametrize("C,BR", [s for s in cases.MRCNN_SHAPES if s[1] < 32768])
def test_oracle_mrcnn_losses_vs_f64(C, BR):
    ids, lg, act, tb, pb = cases.mrcnn_case(C, BR)
    pa, cl, cb, bl, bb = ref.mrcnn_losses_f64(ids, lg, act, tb, pb)
    o_pa, o_cl, o_bl = oracle.mrcnn_losses(ids, lg, act, tb, pb)
    assert np.array_equal(o_pa, pa)
    ref.assert_loss(o_cl, cl, cb, "class")
    ref.assert_loss(o_bl, bl, bb, "box")


def test_oracle_mrcnn_nan_logits_take_the_first_max():
    """A NaN logit at class 0 keeps the argmax at 0; a NaN at a later class never becomes the argmax (np.argmax
    would return it)."""
    for name, ids, lg, act, tb, pb in cases.mrcnn_special_cases():
        pa, cl, cb, bl, bb = ref.mrcnn_losses_f64(ids, lg, act, tb, pb)
        o_pa, o_cl, o_bl = oracle.mrcnn_losses(ids, lg, act, tb, pb)
        assert np.array_equal(o_pa, pa), name
        ref.assert_loss(o_cl, cl, cb, f"{name} class")
        ref.assert_loss(o_bl, bl, bb, f"{name} box")
    lg = np.array([[[1, np.nan, 5, 2], [np.nan, 1, 2, 3]]], f32)
    pa = oracle.mrcnn_losses(np.zeros((1, 2), np.int32), lg, np.array([[1, 0, 2, 4]], f32), np.zeros((1, 2, 4)),
                             np.zeros((1, 2, 4, 4)))[0]
    assert pa.tolist() == [[2, 1]]
