"""numpy replays of the cheap pre-filters that sit in front of exact decisions in the CUDA kernels, checked against the
exact decision on adversarial inputs (no GPU needed).

Each filter replayed here is correct only under a claim stated in its kernel's source:
- frcnn_mask_kernel (frcnn.cu): an fp32 IoU screen settles every pair farther than kMargin from the threshold; only the
  rest take the fp64 arithmetic of the reference. Claimed for coordinates below kFrcnnScreenMaxSide.
- nms_mask_kernel<true> pass 1 (nms.cu): four fp32 sign bits pick a superset of the pairs with positive intersection.
- rpn_anchor_best_kernel (rpn_targets.cu): fp64 boxes rounded outward to fp32, then the same sign test: a superset of
  the pairs with fp64 intersection > 0.
The replays do what the kernels do, operation for operation, in fp32 (the library is built with -fmad=false and
without fast math: no contraction, no flush to zero). Where the device and numpy differ, the replay takes the device's
side: a NaN produced by device arithmetic is the canonical NaN 0x7fffffff, whose sign bit is clear (a NaN that kept
its sign could only add candidates).
"""
import os
import re
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import oracle  # noqa: E402

f32, f64 = np.float32, np.float64
CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "objectdetection_b200", "csrc")


def _constant(source, pattern):
    with open(os.path.join(CSRC, source)) as f:
        m = re.search(pattern, f.read())
    assert m, f"{pattern} not found in {source}"
    return m.group(1)


def _sub(a, b):
    """a - b in fp32 as the device computes it: NaN results are the canonical (positive) NaN."""
    with np.errstate(all="ignore"):
        d = (np.asarray(a, f32) - np.asarray(b, f32)).astype(f32)
    return np.where(np.isnan(d), f32(np.nan), d)


def _sign(x):
    return np.asarray(x, f32).view(np.uint32) >> np.uint32(31)


def _f_min(a, b):   # (b < a) ? b : a
    return np.where(b < a, b, a)


def _f_max(a, b):   # (a < b) ? b : a
    return np.where(a < b, b, a)


# ----------------------------------------------------------------------------- Faster R-CNN fp32 IoU screen
SCREEN_MAX_SIDE = int(_constant("frcnn.cu", r"constexpr int kFrcnnScreenMaxSide = (\d+);"))
SCREEN_MARGIN = f32(float(_constant("frcnn.cu", r"constexpr float kMargin = ([0-9.e+-]+)f;")))


def frcnn_screen(bi, bj, thr, certain=False):
    """frcnn_mask_kernel's fp32 screen for box i (earlier) and box j (later), [n,4] fp64 (x1,y1,x2,y2).
    Returns (say_hit, say_miss): whether the screen can set / clear the keep bit without the fp64 path (with
    `certain`: whether it does so for every quotient __fdividef may return).
    __fdividef is modelled as the correctly rounded quotient widened by its documented 2-ulp error."""
    def cvt(b):
        area = (b[:, 2] - b[:, 0] + 1) * (b[:, 3] - b[:, 1] + 1)
        return (b[:, 0].astype(f32), b[:, 1].astype(f32), (b[:, 2] + 1).astype(f32), (b[:, 3] + 1).astype(f32),
                area.astype(f32))
    mx1, my1, mx2, my2, ma = cvt(bi)
    cx1, cy1, cx2, cy2, ca = cvt(bj)
    zero = f32(0)
    fw = np.maximum(zero, _sub(np.minimum(mx2, cx2), np.maximum(mx1, cx1)))
    fh = np.maximum(zero, _sub(np.minimum(my2, cy2), np.maximum(my1, cy1)))
    fi = (fw * fh).astype(f32)
    den = _sub((ma + ca).astype(f32), fi)
    fo = (fi / den).astype(f32)
    lo = np.nextafter(np.nextafter(fo, f32(-np.inf)), f32(-np.inf))
    hi = np.nextafter(np.nextafter(fo, f32(np.inf)), f32(np.inf))
    thr_hi, thr_lo = f32(f32(thr) + SCREEN_MARGIN), f32(f32(thr) - SCREEN_MARGIN)
    return (lo > thr_hi, hi < thr_lo) if certain else (hi > thr_hi, lo < thr_lo)


def frcnn_exact(bi, bj, thr):
    """proposals.py:141-164 in fp64: box j is suppressed by box i iff ovr >= thr."""
    xx1, yy1 = np.maximum(bi[:, 0], bj[:, 0]), np.maximum(bi[:, 1], bj[:, 1])
    xx2, yy2 = np.minimum(bi[:, 2], bj[:, 2]), np.minimum(bi[:, 3], bj[:, 3])
    w, h = np.maximum(0.0, xx2 - xx1 + 1), np.maximum(0.0, yy2 - yy1 + 1)
    inter = w * h
    ai = (bi[:, 2] - bi[:, 0] + 1) * (bi[:, 3] - bi[:, 1] + 1)
    aj = (bj[:, 2] - bj[:, 0] + 1) * (bj[:, 3] - bj[:, 1] + 1)
    return inter / (ai + aj - inter) >= thr


def near_threshold_pairs(rs, n, thr, lo, hi):
    """n pairs of boxes with sides of 1-4 px (the +1 convention), one corner in [lo, hi) on both axes, clipped like the
    decode kernel clips to an image of side `hi`; box j is box i shifted so that the IoU is within ~1e-2 of thr."""
    side = rs.uniform(1.0, 4.0, (n, 2))
    x1 = rs.uniform(lo, hi - 12.0, (n, 2))
    bi = np.concatenate([x1, x1 + side - 1.0], 1)
    # same-size boxes shifted along one axis by d have IoU (s - d) / (s + d); every corner is then jittered, by up to
    # 5e-3 px for half of the pairs (mostly inside the margin) and up to 2e-2 px for the others
    axis = rs.randint(0, 2, n)
    s = side[np.arange(n), axis]
    d = s * (1 - thr) / (1 + thr)
    bj = bi.copy()
    bj[np.arange(n), axis] += d
    bj[np.arange(n), axis + 2] += d
    bj += rs.uniform(-1, 1, bj.shape) * np.where(rs.random_sample(n) < 0.5, 5e-3, 2e-2)[:, None]
    bj[:, 2:] = np.maximum(bj[:, 2:], bj[:, :2])
    order = rs.random_sample(n) < 0.5                       # either box may be the earlier one
    bi[order], bj[order] = bj[order].copy(), bi[order].copy()
    return np.clip(bi, 0, hi - 1), np.clip(bj, 0, hi - 1)


def _screen_misjudged(bi, bj, thr):
    say_hit, say_miss = frcnn_screen(bi, bj, thr)
    exact = frcnn_exact(bi, bj, thr)
    return (say_hit & ~exact) | (say_miss & exact), say_hit | say_miss


@pytest.mark.parametrize("thr", [0.7, 0.5, 0.2])
def test_frcnn_screen_agrees_with_fp64_over_screened_domain(thr):
    """Near-threshold pairs of the smallest boxes anywhere below kFrcnnScreenMaxSide, half of them in its top half,
    where fp32 rounds coarsest: the screen never decides against the fp64 reference on a pair it settles."""
    rs = np.random.RandomState(int(thr * 100))
    n = 1_000_000
    for lo in (0.0, SCREEN_MAX_SIDE / 2):
        bi, bj = near_threshold_pairs(rs, n, thr, lo, SCREEN_MAX_SIDE)
        bad, settled = _screen_misjudged(bi, bj, thr)
        assert settled.mean() > 0.1        # the screen settles a good share of these pairs: the check has teeth
        assert not bad.any(), (f"{int(bad.sum())} pairs misjudged below {SCREEN_MAX_SIDE} px, first "
                               f"{bi[bad][0].tolist()} vs {bj[bad][0].tolist()}")


def test_frcnn_screen_is_wrong_past_its_bound():
    """Why frcnn.cu sends larger images to the fp64 path: at coordinates near 1.2e5 px the same screen misjudges
    near-threshold pairs of small boxes."""
    rs = np.random.RandomState(3)
    bi, bj = near_threshold_pairs(rs, 1_000_000, 0.7, 110_000, 131_072)
    bad, _ = _screen_misjudged(bi, bj, 0.7)
    assert bad.sum() > 10


# ----------------------------------------------------------------------------- NMS pass 1 (sign bits)
def _adversarial_values():
    tiny = np.float32(1e-45)                                    # smallest subnormal
    one = f32(1.0)
    return dict(tiny=tiny, sub=f32(3e-39), fmin=f32(np.finfo(f32).tiny), one=one,
                one_up=np.nextafter(one, f32(2)), one_dn=np.nextafter(one, f32(0)),
                big=f32(3e38), fmax=np.finfo(f32).max, inf=f32(np.inf), nan=f32(np.nan),
                nneg=np.array([0xFFC00000], np.uint32).view(f32)[0],
                npay=np.array([0x7FC01234], np.uint32).view(f32)[0])


def nms_adversarial_boxes(rs=None):
    """[n,4] float32 (y1,x1,y2,x2): signed zeros, shared edges, one-ulp overlaps, subnormal sides, infinities, NaN (both
    signs, two payloads) in each of the four positions, flipped boxes and magnitudes whose differences overflow, plus
    random boxes built from those values."""
    v = _adversarial_values()
    z, nz, one, up, dn = f32(0.0), f32(-0.0), v["one"], v["one_up"], v["one_dn"]
    rows = [
        [z, z, one, one], [nz, nz, one, one], [z, nz, one, one], [one, one, z, z],            # +-0, flipped
        [z, one, one, f32(2)], [one, z, f32(2), one], [z, dn, one, f32(2)], [z, up, one, f32(2)],  # shared edge, 1 ulp
        [dn, z, f32(2), one], [up, z, f32(2), one], [z, z, up, up], [z, z, dn, dn],
        [z, z, v["tiny"], one], [z, z, one, v["tiny"]], [nz, nz, v["tiny"], v["tiny"]],        # subnormal sides
        [z, z, v["sub"], v["sub"]], [v["tiny"], z, one, one], [-v["tiny"], -v["tiny"], v["fmin"], v["fmin"]],
        [-v["inf"], -v["inf"], v["inf"], v["inf"]], [z, z, v["inf"], v["inf"]], [-v["inf"], z, z, one],
        [v["inf"], v["inf"], v["inf"], v["inf"]], [z, -v["inf"], one, one],
        [-v["big"], -v["big"], v["big"], v["big"]], [v["big"], v["big"], -v["big"], -v["big"]],
        [-v["fmax"], z, v["fmax"], one], [z, -v["fmax"], one, v["fmax"]], [-v["big"], -v["big"], z, z],
        [v["big"], z, v["fmax"], one], [-v["fmax"], -v["fmax"], -v["big"], -v["big"]],
        [f32(0.25), f32(0.25), f32(0.75), f32(0.75)], [f32(0.5), f32(0.5), f32(1.5), f32(1.5)],
    ]
    for nan in (v["nan"], v["nneg"], v["npay"]):                # NaN in each position of a box overlapping the others
        for p in range(4):
            b = [z, z, one, one]
            b[p] = nan
            rows.append(b)
    pool = np.array([z, nz, one, up, dn, f32(2), f32(0.5), v["tiny"], -v["tiny"], v["sub"], v["fmin"], v["big"],
                     -v["big"], v["fmax"], -v["fmax"], v["inf"], -v["inf"], v["nan"], v["nneg"]], f32)
    rs = rs or np.random.RandomState(0)
    rand = pool[rs.randint(0, pool.size, (96, 4))]
    return np.concatenate([np.array(rows, f32), rand]).astype(f32)


def _canon(b):
    ymin, xmin = _f_min(b[:, 0], b[:, 2]), _f_min(b[:, 1], b[:, 3])
    ymax, xmax = _f_max(b[:, 0], b[:, 2]), _f_max(b[:, 1], b[:, 3])
    with np.errstate(all="ignore"):
        area = ((ymax - ymin) * (xmax - xmin)).astype(f32)
    return ymin, xmin, ymax, xmax, area


def nms_candidates(boxes):
    """Pass 1 of nms_mask_kernel<true> for every ordered pair: [i, j] = row box i (`my`), column box j (`c`)."""
    ymin, xmin, ymax, xmax, _ = _canon(boxes)
    r, c = (slice(None), None), (None, slice(None))
    sgn = (_sign(_sub(ymin[c], ymax[r])) & _sign(_sub(ymin[r], ymax[c])) &
           _sign(_sub(xmin[c], xmax[r])) & _sign(_sub(xmin[r], xmax[c])))
    return sgn.astype(bool)


def nms_pass2(boxes, thr):
    """Pass 2 of nms_mask_kernel<true> (the exact TF IoU in the kernel's operand order, `inter > 0` guard)."""
    ymin, xmin, ymax, xmax, area = _canon(boxes)
    r, c = (slice(None), None), (None, slice(None))
    with np.errstate(all="ignore"):
        ih = _sub(_f_min(ymax[r], ymax[c]), _f_max(ymin[r], ymin[c]))
        iw = _sub(_f_min(xmax[r], xmax[c]), _f_max(xmin[r], xmin[c]))
        inter = (_f_max(ih, f32(0)) * _f_max(iw, f32(0))).astype(f32)
        den = ((area[r] + area[c]).astype(f32) - inter).astype(f32)
        return (inter > 0) & ((inter / den).astype(f32) > f32(thr))


@pytest.mark.parametrize("thr", [0.0, 1e-7, 0.5, 1.0])
def test_nms_sign_bit_candidates_cover_every_suppression(thr):
    """Every pair whose TF IoU (the oracle's tf_iou) exceeds thr is a pass-1 candidate, and pass 1 + pass 2 decide
    every pair exactly as tf_iou(later, earlier) > thr, the comparison the oracle's greedy loop makes."""
    boxes = nms_adversarial_boxes()
    n = boxes.shape[0]
    cand = nms_candidates(boxes)
    decided = cand & nms_pass2(boxes, thr)
    want = np.zeros((n, n), bool)
    for i in range(n):
        for j in range(n):
            if i != j:
                want[i, j] = oracle.tf_iou(boxes[j], boxes[i]) > f32(thr)
    np.fill_diagonal(decided, False)
    missed = want & ~cand
    assert not missed.any(), [(boxes[i].tolist(), boxes[j].tolist()) for i, j in np.argwhere(missed)[:3]]
    assert np.array_equal(decided, want), np.argwhere(decided != want)[:5].tolist()
    if thr < 1.0:
        assert want.sum() > 20          # the set has suppressing pairs for every threshold below 1


def test_nms_adversarial_set_reaches_the_edges():
    """The box set contains what it claims: one-ulp overlaps that are candidates, shared edges that are not, and
    differences that overflow to infinity."""
    boxes = nms_adversarial_boxes()
    cand = nms_candidates(boxes)
    # in x, [1-ulp,2] overlaps [0,1] by one ulp, [1,2] only touches it and [1+ulp,2] is one ulp away
    assert cand[0, 6] and not cand[0, 4] and not cand[0, 7]
    ymin, _, ymax, _, _ = _canon(boxes)
    with np.errstate(all="ignore"):
        assert np.isinf(ymin[:, None] - ymax[None, :]).any() and np.isnan(boxes).any()


# ----------------------------------------------------------------------------- RPN targets: outward rounding
def _round_f32(x, down):
    """__double2float_rd (down) / __double2float_ru: the fp32 value next to x on the given side."""
    x = np.asarray(x, f64)
    with np.errstate(over="ignore"):
        f = x.astype(f32)
    fx = f.astype(f64)
    if down:
        return np.where(fx > x, np.nextafter(f, f32(-np.inf)), f).astype(f32)
    return np.where(fx < x, np.nextafter(f, f32(np.inf)), f).astype(f32)


def conservative_f32(b):
    """rpn_targets.cu conservative_f32: [n,4] fp64 (y1,x1,y2,x2) -> fp32 with mins rounded down, maxes up."""
    return np.stack([_round_f32(b[:, 0], True), _round_f32(b[:, 1], True),
                     _round_f32(b[:, 2], False), _round_f32(b[:, 3], False)], 1)


def may_overlap(a, g):
    """rpn_targets.cu may_overlap for anchors a [A,4] x GT g [G,4] (fp32 conservative copies) -> [A,G]."""
    A, G = a[:, None, :], g[None, :, :]
    return (_sign(_sub(G[..., 0], A[..., 2])) & _sign(_sub(A[..., 0], G[..., 2])) &
            _sign(_sub(G[..., 1], A[..., 3])) & _sign(_sub(A[..., 1], G[..., 3]))).astype(bool)


def rpn_inter(a, g):
    """rpn_iou's fp64 intersection (CUDA fmax/fmin: NaN-ignoring, like np.fmax/np.fmin) -> [A,G]."""
    A, G = a[:, None, :], g[None, :, :]
    y1, y2 = np.fmax(G[..., 0], A[..., 0]), np.fmin(G[..., 2], A[..., 2])
    x1, x2 = np.fmax(G[..., 1], A[..., 1]), np.fmin(G[..., 3], A[..., 3])
    return np.fmax(x2 - x1, 0.0) * np.fmax(y2 - y1, 0.0)


def rpn_near_resolution_boxes(rs, m):
    """Anchors and GT boxes with edges at magnitude m whose fp64 distances are below fp32's resolution there: slivers of
    overlap from one fp64 ulp up to a few fp32 ulps on each axis, touching edges and zero-width GT boxes."""
    u32 = float(np.spacing(f32(m)))
    eps = np.array([np.spacing(f64(m)), 1e-6 * u32, 0.25 * u32, 0.5 * u32, 0.75 * u32, u32, 1.5 * u32, 3 * u32])
    L = max(64 * u32, 4.0)
    base = np.array([m, m, m + L, m + L])
    anchors, gts = [], []
    for e in np.concatenate([eps, -eps, [0.0]]):            # e > 0 overlap, e < 0 gap, 0 touching
        for axis in (0, 1):
            a = base.copy()
            g = base.copy()
            g[axis], g[axis + 2] = a[axis + 2] - e, a[axis + 2] - e + L   # g starts e before a ends
            anchors.append(a)
            gts.append(g)
            g0 = g.copy()
            g0[axis + 2] = g0[axis]                        # zero-width GT on the same edge
            gts.append(g0)
    jitter = rs.uniform(-3 * u32, 3 * u32, (200, 4))       # dense random edges straddling a few fp32 values
    rand = np.array([m, m, m + L, m + L]) + jitter
    rand[:, 2:] = np.maximum(rand[:, 2:], rand[:, :2])
    anchors, gts = np.array(anchors + list(rand[:100])), np.array(gts + list(rand[100:]))
    sign = np.where(rs.random_sample(anchors.shape[0]) < 0.25, -1.0, 1.0)[:, None]
    anchors[sign[:, 0] < 0] = -anchors[sign[:, 0] < 0][:, [2, 3, 0, 1]]    # mirrored to -m as well
    return anchors, gts


@pytest.mark.parametrize("m", [1e3, 2.0 ** 24, 1e7, -1e3])
def test_rpn_outward_rounding_covers_every_overlap(m):
    """may_overlap on the outward-rounded fp32 copies holds for every pair whose fp64 intersection is positive."""
    rs = np.random.RandomState(int(abs(m)) % 1000)
    anchors, gts = rpn_near_resolution_boxes(rs, m)
    inter = rpn_inter(anchors, gts)
    cand = may_overlap(conservative_f32(anchors), conservative_f32(gts))
    missed = (inter > 0) & ~cand
    assert not missed.any(), [(anchors[i].tolist(), gts[j].tolist()) for i, j in np.argwhere(missed)[:3]]
    # the set holds overlaps that fp32 cannot see with round-to-nearest copies
    near = lambda b: b.astype(f32)    # noqa: E731
    assert ((inter > 0) & ~may_overlap(near(anchors), near(gts))).any()


def test_rpn_outward_rounding_beyond_fp32_range():
    """Edges beyond fp32's range round to +-FLT_MAX / +-inf and still order correctly."""
    big = np.array([[-1e39, -1e39, 1e39, 1e39], [1e39, 0.0, 2e39, 1.0], [0.0, 0.0, 1.0, 1.0], [-2e39, 0.0, -1e39, 1.0],
                    [-np.inf, -np.inf, np.inf, np.inf], [3.5e38, 0.0, 3.6e38, 1.0], [1.5e39, 0.5, 1.6e39, 0.75]])
    with np.errstate(invalid="ignore"):
        inter = rpn_inter(big, big)
    cand = may_overlap(conservative_f32(big), conservative_f32(big))
    missed = (inter > 0) & ~cand
    assert not missed.any(), np.argwhere(missed).tolist()
