"""The two outputs that no reference-run golden pins - the mask targets of od_detection_target_forward
(mask_target_kernel) and the forward values of the four head losses (csrc/losses.cu) - checked on the GPU against the
independent float64 restatements of tests/_f64_refs.py, and against the oracle wherever the older tests compare bit for
bit. The cases sit where these kernels could go wrong unnoticed: GT lists whose class-0 rows are not all at the end (the
compacted-to-original GT mapping), mask sizes of 1, exact rounding ties, ROIs outside their GT box, R at the 4096 cap;
chunk tails and borders of the RPN loss, empty images between images with positives, non-finite and overflowing
values, argmax ties and NaN logits, the BCE clip.

Mask targets are compared exactly on every pixel the float64 reference can decide (undecidable pixels must be 0 or 1,
and at least 95 % of the pixels of every case must be decidable); losses within the error budget of the reference.
The input builders are plain functions so that tests/test_f64_refs.py runs the oracle on the same inputs without a
GPU."""
import ctypes
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import _f64_refs as ref  # noqa: E402
import _synth  # noqa: E402

import oracle  # noqa: E402
from objectdetection_b200.config import config as Conf  # noqa: E402

torch = pytest.importorskip("torch")
f32 = np.float32


# ------------------------------------------------------------------ inputs
def _blob_masks(rs, B, Mh, Mw, G, soft=False):
    """[B,Mh,Mw,G] ellipse masks; soft: a smooth ramp in [0, 1] instead of 0/1."""
    yy, xx = np.mgrid[0:Mh, 0:Mw]
    masks = np.zeros((B, Mh, Mw, G), f32)
    for b in range(B):
        for g in range(G):
            cy, cx = rs.uniform(0.2, 0.8) * Mh, rs.uniform(0.2, 0.8) * Mw
            ry, rx = rs.uniform(0.15, 0.45) * Mh, rs.uniform(0.15, 0.45) * Mw
            r2 = ((yy - cy) / ry) ** 2 + ((xx - cx) / rx) ** 2
            masks[b, :, :, g] = np.clip(1.5 - r2, 0, 1) if soft else (r2 < 1)
    return masks


def _pad_gt(rs, cls, gt, where):
    """Move the class-0 (padding) rows of every image to the start, the middle or interleave them with the valid rows."""
    B, G = cls.shape
    for b in range(B):
        valid = np.nonzero(cls[b] != 0)[0]
        nv = valid.size
        if where == "start":
            rows = np.arange(G - nv, G)
        elif where == "middle":
            rows = np.concatenate([np.arange(nv // 2), np.arange(G - (nv - nv // 2), G)])
        else:
            rows = np.sort(rs.choice(G, nv, replace=False))
        c, g = np.zeros_like(cls[b]), np.zeros_like(gt[b])
        c[rows], g[rows] = cls[b, valid], gt[b, valid]
        g[c == 0] = rs.uniform(0, 1, (G - nv, 4))          # padding rows hold junk boxes: class 0 alone marks them
        cls[b], gt[b] = c, g


def mask_case(name):
    """(mask_shape, rois_per_image, props, cls, gt, pp, pn, masks [B,Mh,Mw,G]) of one named mask-target case."""
    rs = np.random.RandomState(sum(map(ord, name)))
    shape, R = (28, 28), 200
    if name in ("pad_start", "pad_middle", "pad_interleaved"):
        props, cls, gt, pp, pn = _synth.target_inputs(rs, 8, 2000, 100)
        for b in range(8):                                  # 20 to 60 valid GT rows of 100
            nv = rs.randint(20, 61)
            src = rs.choice(1800, nv, replace=False)
            gt[b, :nv] = props[b, src] + rs.normal(0, 0.01, (nv, 4)).astype(f32)
            cls[b, :nv] = rs.randint(1, 81, nv)
            cls[b, nv:] = 0
        _pad_gt(rs, cls, gt, name[4:])
        masks = _blob_masks(rs, 8, 56, 40, 100)
    elif name.startswith("shape_"):
        shape = tuple(int(v) for v in name[6:].split("x"))
        props, cls, gt, pp, pn = _synth.target_inputs(rs, 2, 600, 20, n_pad=100)
        _pad_gt(rs, cls, gt, "interleaved")
        masks = _blob_masks(rs, 2, 56, 40, 20)
    elif name == "full_image_1024":
        props, cls, gt, pp, pn = _synth.target_inputs(rs, 2, 500, 6, n_pad=50)
        masks = np.zeros((2, 1024, 1024, 6), f32)
        for b in range(2):
            for g in range(6):
                y1, x1, y2, x2 = np.clip(np.round(gt[b, g] * 1023), 0, 1023).astype(int)
                masks[b, y1:y2 + 1, x1:x2 + 1, g] = 1
                masks[b, (y1 + y2) // 2:y2 + 1, x1:(x1 + x2) // 2, g] = 0          # a notch in each object
    elif name == "exact_tie":
        # the CPU known answer on the device: box [0,0,1,1] over a 3x3 mask with columns [0,1,0], 5x5 targets: the taps
        # at x = 0.5 and 1.5 give exactly 0.5, which rounds to 0 (half to even)
        shape = (5, 5)
        props = np.zeros((1, 64, 4), f32)
        props[0, :40] = _synth.random_boxes(rs, 40) * f32(0.2) + f32(0.8)
        props[0, 3] = [0, 0, 1, 1]
        gt = np.zeros((1, 4, 4), f32)
        gt[0, 1] = [0, 0, 1, 1]
        cls = np.array([[0, 5, 0, 0]], np.int32)
        pp = pn = np.arange(64, dtype=np.int32)[None]
        masks = np.zeros((1, 3, 3, 4), f32)
        masks[0, :, 1, :] = 1
    elif name == "roi_vs_gt_box":
        # ROIs equal to, larger than (x1.3 about the centre, IoU 0.59) and partly outside (shifted by a fifth) their GT box
        G = 12
        props = np.zeros((2, 400, 4), f32)
        gt = np.zeros((2, G, 4), f32)
        cls = np.zeros((2, G), np.int32)
        for b in range(2):
            c = rs.uniform(0.25, 0.75, (G, 2))
            hw = rs.uniform(0.08, 0.3, (G, 2))
            gt[b] = np.concatenate([c - hw / 2, c + hw / 2], 1)
            cls[b] = rs.randint(1, 81, G)
            big = np.concatenate([c - 0.65 * hw, c + 0.65 * hw], 1)
            sh = gt[b] + np.concatenate([hw, hw], 1) * rs.choice([-0.2, 0.2], (G, 4))
            props[b, :3 * G] = np.concatenate([gt[b], big, sh])
            props[b, 3 * G:360] = _synth.random_boxes(rs, 360 - 3 * G)
        cls[:, ::5] = 0
        pp = np.stack([rs.permutation(400) for _ in range(2)]).astype(np.int32)
        pn = pp.copy()
        masks = _blob_masks(rs, 2, 28, 36, G)
    elif name == "thin_gt":
        # GT boxes one ulp high or wide (the closest to gt_h = 0 that a positive can reach: a GT box of zero height has
        # IoU 0 with every proposal) next to zero-height and zero-width GT rows that no ROI is assigned to
        G = 8
        props = np.zeros((1, 100, 4), f32)
        gt = np.zeros((1, G, 4), f32)
        y, x = f32(0.5), f32(0.25)
        gt[0, 0] = [y, 0.1, np.nextafter(y, f32(1)), 0.6]
        gt[0, 1] = [0.1, x, 0.7, np.nextafter(x, f32(1))]
        gt[0, 2] = [0.3, 0.2, 0.3, 0.7]
        gt[0, 3] = [0.2, 0.4, 0.8, 0.4]
        gt[0, 4:] = _synth.random_boxes(rs, 4)
        cls = np.array([[3, 4, 5, 6, 7, 8, 9, 0]], np.int32)
        props[0, 0], props[0, 1] = gt[0, 0], gt[0, 1]
        props[0, 2] = [y, 0.15, np.nextafter(y, f32(1)), 0.6]
        props[0, 3:7] = gt[0, 4:8]
        props[0, 7:80] = _synth.random_boxes(rs, 73)
        pp = pn = np.arange(100, dtype=np.int32)[None]
        masks = _blob_masks(rs, 1, 20, 24, G)
    elif name == "soft_masks":
        props, cls, gt, pp, pn = _synth.target_inputs(rs, 3, 600, 20, n_pad=100)
        _pad_gt(rs, cls, gt, "middle")
        masks = _blob_masks(rs, 3, 56, 56, 20, soft=True)
    elif name == "rois_4096":
        # R at the 4096 cap of the mask_src workspace: 1351 positive slots per image, filled from many GT copies
        R = 4096
        N, G = 8000, 200
        props = _synth.rois_log_uniform(rs, 2, N)
        gt = np.zeros((2, G, 4), f32)
        cls = rs.randint(1, 81, (2, G)).astype(np.int32)
        for b in range(2):
            gt[b] = props[b, rs.choice(N, G, replace=False)]
            own = rs.randint(0, G, N // 2)
            props[b, :N // 2] = gt[b, own] + rs.normal(0, 0.001, (N // 2, 4)).astype(f32)
        cls[:, 1::7] = 0
        pp = np.stack([rs.permutation(N) for _ in range(2)]).astype(np.int32)
        pn = np.stack([rs.permutation(N) for _ in range(2)]).astype(np.int32)
        masks = _blob_masks(rs, 2, 28, 28, G)
    else:
        raise KeyError(name)
    return shape, R, props, cls, gt, pp, pn, masks


MASK_CASES = ["pad_start", "pad_middle", "pad_interleaved", "shape_14x28", "shape_1x1", "shape_1x5", "shape_5x1",
              "full_image_1024", "exact_tie", "roi_vs_gt_box", "thin_gt", "soft_masks", "rois_4096"]


def check_masks_against_f64(shape, mini, props, cls, gt, masks, rois, n_pos, assignment, targets):
    """targets [B,R,mh,mw] of a run (kernel or oracle) against mask_targets_f64: exact on decidable pixels, 0 or 1
    elsewhere, zero rows past the positives. assignment [B,R] (compacted GT index, the debug output) must equal the
    float64 first-max argmax on the rows whose best IoU is not tied. Returns the decidable fraction."""
    dec_n = tot_n = 0
    for b in range(props.shape[0]):
        P = int(n_pos[b])
        assert not targets[b, P:].any(), b
        if P == 0:
            continue
        rows, comp, amb = ref.gt_assignment_f64(rois[b, :P], gt[b], cls[b])
        if assignment is not None:
            bad = (assignment[b, :P] != comp) & ~amb
            assert not bad.any(), (b, np.nonzero(bad)[0][:5], assignment[b, :P][bad][:5], comp[bad][:5])
        value, dec = ref.mask_targets_f64(rois[b, :P], gt[b], rows, masks[b], shape, mini)
        dec &= ~amb[:, None, None]
        got = targets[b, :P]
        want = np.round(value)
        bad = dec & (got != want)
        assert not bad.any(), (b, np.argwhere(bad)[:5].tolist(), got[bad][:5], value[bad][:5])
        assert np.isin(got[~dec], [0.0, 1.0]).all(), b
        dec_n += int(dec.sum())
        tot_n += dec.size
    assert tot_n > 0, "no positive ROI"
    assert dec_n >= 0.95 * tot_n, f"only {dec_n} of {tot_n} pixels decidable"
    return dec_n / tot_n


# ------------------------------------------------------------------ device calls
def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    torch.cuda.synchronize()
    return t.detach().cpu().numpy()


@pytest.fixture(scope="module")
def _cuda():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (there is no CPU path)")


def _targets(shape, R, mini, props, cls, gt, pp, pn, masks, layout_hwg):
    """od_detection_target_forward with masks in the [B,Mh,Mw,G] (layout_hwg) or [B,G,Mh,Mw] layout and the debug
    outputs counts and gt_assignment. Returns (rois, mask_targets, counts, gt_assignment) on the host."""
    from objectdetection_b200 import _lib
    B, N = props.shape[:2]
    G = cls.shape[1]
    if not layout_hwg:
        masks = masks.transpose(0, 3, 1, 2)
    t = {k: cu(v) for k, v in dict(props=props, cls=cls, gt=gt, pp=pp, pn=pn, masks=masks).items()}
    rois = torch.empty((B, R, 4), dtype=torch.float32, device="cuda")
    rcls = torch.empty((B, R), dtype=torch.int32, device="cuda")
    deltas = torch.empty((B, R, 4), dtype=torch.float32, device="cuda")
    targets = torch.full((B, R) + tuple(shape), -1.0, dtype=torch.float32, device="cuda")
    counts = torch.empty((B, 6), dtype=torch.int32, device="cuda")
    assign = torch.empty((B, R), dtype=torch.int32, device="cuda")
    params = _lib.TargetParams(R, (ctypes.c_float * 4)(*Conf.BBOX_STD_DEV), shape[0], shape[1], 1 if mini else 0,
                               1 if layout_hwg else 0)
    L = _lib.lib()
    dl = _lib.DL()
    dbg = _lib.TargetDebug()
    dbg.counts, dbg.gt_assignment = dl(counts), dl(assign)
    ws = _lib.workspace(L.od_detection_target_workspace_bytes(B, N, G), rois.device)
    _lib.check(L.od_detection_target_forward(dl(t["props"]), dl(t["cls"]), dl(t["gt"]), dl(t["pp"]), dl(t["pn"]),
                                             ctypes.byref(params), dl(rois), dl(rcls), dl(deltas), dl(t["masks"]),
                                             dl(targets), ctypes.byref(dbg), ws.data_ptr(), ws.numel(),
                                             _lib.stream_ptr(rois.device)), "od_detection_target_forward")
    return host(rois), host(targets), host(counts), host(assign)


# ------------------------------------------------------------------ mask targets
@pytest.mark.gpu
@pytest.mark.parametrize("mini", [True, False])
@pytest.mark.parametrize("case", MASK_CASES)
def test_mask_targets_f64(_cuda, case, mini):
    shape, R, props, cls, gt, pp, pn, masks = mask_case(case)
    rois, got, counts, assign = _targets(shape, R, mini, props, cls, gt, pp, pn, masks, True)
    rois0, got0, _, _ = _targets(shape, R, mini, props, cls, gt, pp, pn, masks, False)
    assert np.array_equal(got0, got) and np.array_equal(rois0, rois), "the two mask layouts disagree"
    n_pos = counts[:, 4]
    frac = check_masks_against_f64(shape, mini, props, cls, gt, masks, rois, n_pos, assign, got)
    for b in range(props.shape[0]):
        w_rois, _, _, wd = oracle.detection_targets(props[b], cls[b], gt[b], pp[b], pn[b], R, Conf.BBOX_STD_DEV)
        assert np.array_equal(rois[b].view(np.uint32), w_rois.view(np.uint32)), b
        want = oracle.mask_targets(w_rois, cls[b], gt[b], masks[b], wd, shape, mini)
        assert np.array_equal(got[b], want), (b, np.argwhere(got[b] != want)[:5].tolist())
    if case == "exact_tie":
        assert n_pos[0] >= 1 and np.array_equal(got[0, 0], np.tile([0, 0, 1, 0, 0], (5, 1)))
    if case == "rois_4096":
        assert (n_pos == 1351).all(), n_pos
    print(f"{case} mini={mini}: positives {n_pos.tolist()}, decidable {frac:.4f}")


# ------------------------------------------------------------------ RPN losses
RPN_SHAPES = [(A, B) for A in (1, 3, 1023, 1024, 1025, 4097, 261888) for B in (1, 3, 8)]


def rpn_case(A, B):
    """Targets in {-1, 0, 1, 2, -7} ([B,A] or [B,A,1]), positives at anchors 0, 1023, 1024 and A-1, image 1 without
    positives, T in {0, 1, all positives of an image, fewer than one image's positives}; logits with rows at +-80,
    +-1e4, equal pairs and -inf on the non-label side; box differences at 1, nextafter(1, 0) and beyond."""
    rs = np.random.RandomState(A * 10 + B)
    tc = rs.choice([-1, 0, 1, 2, -7], size=(B, A), p=[.3, .55, .1, .03, .02]).astype(np.int32)
    for i in (0, 1023, 1024, A - 1):
        if 0 <= i < A:
            tc[0, i] = 1
            tc[-1, i] = 1
    if B >= 3:
        tc[1][tc[1] == 1] = 0
    npos = (tc == 1).sum(1)
    T = [0, 1, int(npos.max()), max(int(npos.max()) // 2, 1)][(A + B) % 4]
    lg = rs.normal(0, 2, (B, A, 2)).astype(f32)
    k = min(A, 40)
    rows = rs.choice(A, k, replace=False)
    special = np.array([[80, -80], [-80, 80], [1e4, -1e4], [-1e4, 1e4], [3.5, 3.5], [-1e4, -1e4]], f32)
    lg[0, rows] = special[np.arange(k) % len(special)]
    lab = tc[0, rows[:3]] == 1                               # -inf on the non-label side: CE exactly 0
    lg[0, rows[:3], np.where(lab, 0, 1)] = -np.inf
    lg[0, rows[:3], np.where(lab, 1, 0)] = 2.0
    tb = rs.normal(0, 1, (B, T, 4)).astype(f32)
    pb = rs.normal(0, 1.5, (B, A, 4)).astype(f32)
    if T:                                                    # anchor 0 is image 0's first positive: it pairs with row 0
        tb[0, 0] = 0
        pb[0, 0] = [1, -1, np.nextafter(f32(1), f32(0)), 1e6]
    if (A + B) % 2:
        tc = tc[..., None]
    return tc, lg, tb, pb


def _rpn_kernel(tc, lg, tb, pb, pos_rows):
    """od_rpn_loss_forward; pred_box_pos has pos_rows rows pre-filled with -3. Returns (losses, pred_box_pos, num)."""
    from objectdetection_b200 import _lib
    L, dl = _lib.lib(), _lib.DL()
    B, A = lg.shape[:2]
    t = [cu(v) for v in (tc, lg, tb, pb)]
    out = torch.full((2,), -1.0, dtype=torch.float32, device="cuda")
    pos = torch.full((pos_rows, 4), -3.0, dtype=torch.float32, device="cuda")
    num = torch.zeros((1,), dtype=torch.int32, device="cuda")
    ws = _lib.workspace(L.od_rpn_loss_workspace_bytes(B, A), out.device)
    _lib.check(L.od_rpn_loss_forward(dl(t[0]), dl(t[1]), dl(t[2]), dl(t[3]), dl(out), dl(pos), dl(num), ws.data_ptr(),
                                     ws.numel(), _lib.stream_ptr(out.device)), "od_rpn_loss_forward")
    return host(out), host(pos), int(host(num)[0])


@pytest.mark.gpu
@pytest.mark.parametrize("A,B", RPN_SHAPES)
def test_rpn_losses_f64(_cuda, A, B):
    tc, lg, tb, pb = rpn_case(A, B)
    cl, cb, bl, bb, want_pos = ref.rpn_losses_f64(tc, lg, tb, pb)
    n = want_pos.shape[0]
    rows = max(n - 3, 0) if A % 2 else n + 5                  # pred_box_pos shorter and longer than the positives
    got, pos, num = _rpn_kernel(tc, lg, tb, pb, rows)
    ref.assert_loss(got[0], cl, cb, "rpn class loss")
    ref.assert_loss(got[1], bl, bb, "rpn box loss")
    assert num == n
    k = min(rows, n)
    assert np.array_equal(pos[:k], want_pos[:k]) and (pos[k:] == -3.0).all()
    w_cls, w_box, w_pos = oracle.rpn_losses(tc, lg, tb, pb)
    assert np.isclose(got[0], w_cls, rtol=1e-6) and np.isclose(got[1], w_box, rtol=1e-6)
    again, _, _ = _rpn_kernel(tc, lg, tb, pb, rows)
    assert np.array_equal(again.view(np.uint32), got.view(np.uint32)), "two identical calls differ"


def rpn_nonfinite_cases():
    """(name, tc, lg, tb, pb): one row each at a logit gap beyond the fp32 range, +inf, NaN, and box differences whose
    square overflows fp32; 1025 anchors so that the row sits in the second chunk."""
    rs = np.random.RandomState(5)
    out = []
    for name, row, box in (("gap", [3e38, -3e38], None), ("pinf", [np.inf, 0.0], None), ("nan", [np.nan, 1.0], None),
                           ("ninf_label", [5.0, -np.inf], None), ("d_2e19", None, 2e19), ("d_inf", None, 3e38)):
        tc = np.zeros((2, 1025), np.int32)
        tc[:, rs.choice(1025, 200, replace=False)] = 1
        tc[0, 1024] = 1
        lg = rs.normal(0, 1, (2, 1025, 2)).astype(f32)
        tb = rs.normal(0, 1, (2, 300, 4)).astype(f32)
        pb = rs.normal(0, 1, (2, 1025, 4)).astype(f32)
        if row is not None:
            lg[0, 1024] = row
        if box is not None:
            r = int((tc[0, :1024] == 1).sum())
            tb[0, r, 2] = box / 2
            pb[0, 1024, 2] = -box / 2
        out.append((name, tc, lg, tb, pb))
    return out


@pytest.mark.gpu
def test_rpn_losses_non_finite(_cuda):
    """The reference's fp32 graph: a logit gap past the fp32 range gives +inf, a +inf or NaN logit NaN, a -inf label
    logit +inf; |d| = 2e19 overflows d*d and 0 * inf makes the box loss NaN (also when d itself overflows)."""
    expect = dict(gap=(np.inf, None), pinf=(np.nan, None), nan=(np.nan, None), ninf_label=(np.inf, None),
                  d_2e19=(None, np.nan), d_inf=(None, np.nan))
    for name, tc, lg, tb, pb in rpn_nonfinite_cases():
        cl, cb, bl, bb, _ = ref.rpn_losses_f64(tc, lg, tb, pb)
        got, _, _ = _rpn_kernel(tc, lg, tb, pb, 1)
        ec, eb = expect[name]
        if ec is not None:
            assert (np.isnan(cl) and np.isnan(ec)) or cl == ec, (name, cl)
        if eb is not None:
            assert np.isnan(bl), (name, bl)
        ref.assert_loss(got[0], cl, cb, f"{name} class")
        ref.assert_loss(got[1], bl, bb, f"{name} box")


# ------------------------------------------------------------------ mrcnn losses
MRCNN_SHAPES = [(C, BR) for C in (1, 2, 81, 1000) for BR in (1, 1023, 1024, 1025)] + [(2, 32768), (81, 32768)]
_BR = {1: (1, 1), 1023: (3, 341), 1024: (8, 128), 1025: (5, 205), 32768: (8, 4096)}


def mrcnn_case(C, BR):
    """Labels in [0, C) (a third 0), logits quantised to halves so that argmax ties are common, 0/1 active flags with
    class 0 active, BCE predictions at 0, 1, 1e-9, 1 - 1e-8, negative and above 1, targets at 0, 1, 0.5 and outside
    [0, 1]."""
    B, R = _BR[BR]
    rs = np.random.RandomState(C * 7 + BR)
    ids = np.where(rs.random_sample((B, R)) < 1 / 3, 0, rs.randint(0, C, (B, R))).astype(np.int32)
    lg = (np.round(rs.normal(0, 2, (B, R, C)) * 2) / 2).astype(f32)
    act = (rs.random_sample((B, C)) > 0.4).astype(f32)
    act[:, 0] = 1
    tb = rs.random_sample((B, R, 4)).astype(f32)
    pb = rs.random_sample((B, R, C, 4)).astype(f32)
    edges = np.array([0, 1, 1e-9, 1 - 1e-8, -0.5, 1.5, 0.5, 1e-7], f32)
    tedges = np.array([0, 1, 0.5, -0.25, 1.75], f32)
    pos = np.argwhere(ids > 0)
    for k, (b, r) in enumerate(pos[:64]):
        pb[b, r, ids[b, r]] = np.roll(edges, k)[:4]
        tb[b, r] = np.roll(tedges, k)[:4]
    return ids, lg, act, tb, pb


def _mrcnn_kernel(ids, lg, act, tb, pb):
    from objectdetection_b200.loss_optimize import Loss
    pa, c, b = Loss.mrcnn_losses(cu(ids), cu(lg), cu(act), cu(tb), cu(pb))
    return host(pa), float(host(c)), float(host(b))


@pytest.mark.gpu
@pytest.mark.parametrize("C,BR", MRCNN_SHAPES)
def test_mrcnn_losses_f64(_cuda, C, BR):
    ids, lg, act, tb, pb = mrcnn_case(C, BR)
    w_pa, cl, cb, bl, bb = ref.mrcnn_losses_f64(ids, lg, act, tb, pb)
    pa, c, b = _mrcnn_kernel(ids, lg, act, tb, pb)
    assert np.array_equal(pa, w_pa), np.argwhere(pa != w_pa)[:5].tolist()
    ref.assert_loss(c, cl, cb, "mrcnn class loss")
    ref.assert_loss(b, bl, bb, "mrcnn box loss")
    o_pa, o_c, o_b = oracle.mrcnn_losses(ids, lg, act, tb, pb)
    assert np.array_equal(pa, o_pa) and np.isclose(c, o_c, rtol=1e-6, equal_nan=True) and np.isclose(b, o_b, rtol=1e-6)
    again = _mrcnn_kernel(ids, lg, act, tb, pb)
    assert np.array_equal(np.float32(again[1:]).view(np.uint32), np.float32((c, b)).view(np.uint32)), \
        "two identical calls differ"


def mrcnn_special_cases():
    """(name, ids, lg, act, tb, pb) with NaN logits (at class 0 and at a later class), NaN BCE predictions and
    all-inactive predicted classes."""
    out = []
    for name in ("nan_logit_first", "nan_logit_later", "nan_pred", "all_inactive"):
        ids, lg, act, tb, pb = mrcnn_case(81, 1025)
        if name == "nan_logit_first":
            lg[0, :20, 0] = np.nan
        elif name == "nan_logit_later":
            lg[1, :20, 7] = np.nan
            lg[1, 20:40, 80] = np.nan
        elif name == "nan_pred":
            b, r = np.argwhere(ids > 0)[0]
            pb[b, r, ids[b, r], 1] = np.nan
        else:
            act[0] = 0
        out.append((name, ids, lg, act, tb, pb))
    return out


@pytest.mark.gpu
def test_mrcnn_losses_nan_and_inactive(_cuda):
    """NaN logits: pred_active exact (the strict first-max scan keeps a NaN at class 0 and never picks a later one),
    class loss NaN. A NaN prediction makes the box loss NaN; no active predicted class makes the class loss 0/0 = NaN."""
    for name, ids, lg, act, tb, pb in mrcnn_special_cases():
        w_pa, cl, cb, bl, bb = ref.mrcnn_losses_f64(ids, lg, act, tb, pb)
        pa, c, b = _mrcnn_kernel(ids, lg, act, tb, pb)
        assert np.array_equal(pa, w_pa), (name, np.argwhere(pa != w_pa)[:5].tolist())
        assert np.array_equal(pa, oracle.mrcnn_losses(ids, lg, act, tb, pb)[0]), name
        assert np.isnan(cl) == (name != "nan_pred") and np.isnan(bl) == (name == "nan_pred"), name
        ref.assert_loss(c, cl, cb, f"{name} class")
        ref.assert_loss(b, bl, bb, f"{name} box")


@pytest.mark.gpu
def test_mrcnn_losses_out_of_range_labels_pinned(_cuda):
    """Labels -1 and C lie outside the reference's domain. Today the class loss is NaN and their box term is skipped:
    this pins that behaviour so that a change to it is noticed, not judged."""
    ids, lg, act, tb, pb = mrcnn_case(81, 1025)
    bad = ids.copy()
    bad[0, 3], bad[2, 5] = -1, 81
    _, c, b = _mrcnn_kernel(bad, lg, act, tb, pb)
    inside = np.where((bad < 0) | (bad >= 81), 0, bad)
    _, _, _, bl, bb = ref.mrcnn_losses_f64(inside, lg, act, tb, pb)
    assert np.isnan(c)
    ref.assert_loss(b, bl, bb, "box loss without the out-of-range rows")
