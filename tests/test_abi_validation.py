"""Argument validation of every C entry point that takes tensors, table-driven and CPU only.

Each entry point gets one valid baseline call built from hand-made DLTensors (kDLCUDA, small nonzero shapes, fake
256-byte-aligned data pointers, a fake workspace with a large ws_bytes). Every case changes one thing about one
argument and pins the status the call returns, that od_last_error_detail() names the argument, and that a refused call
launched nothing.

The fake pointers are never dereferenced on the host, and all calls run in one child process that sees no GPU
(CUDA_VISIBLE_DEVICES=""): a call that passes validation fails at its first CUDA call with OD_ERR_CUDA (-7) before
anything reaches device memory. So -7 is what an accepted call returns here. The first CUDA call is not always a counted
launch (cudaMemsetAsync, or a kernel started with cudaLaunchKernelEx, fails before the launch is counted), so accepted
calls are recognised by the status alone.
"""
import ctypes
import json
import os
import re
import subprocess
import sys
from ctypes import POINTER, c_int32, c_int64, c_uint8, c_uint16, c_uint64, c_void_p

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
kDLCPU, kDLCUDA = 1, 2
DTYPES = {"f32": (2, 32), "f64": (2, 64), "i32": (0, 32)}
WRONG_DTYPE = (2, 16)          # float16: no entry point takes it
ACCEPTED = -7                  # validation passed, the first CUDA call failed (no GPU is visible)
WS_BYTES = 1 << 40


class _Device(ctypes.Structure):
    _fields_ = [("device_type", c_int32), ("device_id", c_int32)]


class _DType(ctypes.Structure):
    _fields_ = [("code", c_uint8), ("bits", c_uint8), ("lanes", c_uint16)]


class DLTensor(ctypes.Structure):
    _fields_ = [("data", c_void_p), ("device", _Device), ("ndim", c_int32), ("dtype", _DType),
                ("shape", POINTER(c_int64)), ("strides", POINTER(c_int64)), ("byte_offset", c_uint64)]


class Arg:
    """One tensor argument: dtype, baseline shape, the alignment its kernels need (the size of the type they read it as:
    16 for float4, 8 for float2 and double, else 4), whether NULL is accepted, and the extents any value of which is
    valid (`free`)."""

    def __init__(self, name, dtype, shape, align=4, optional=False, free=(), any_strides=False):
        self.name, self.dtype, self.shape, self.align = name, dtype, tuple(shape), align
        self.optional, self.free, self.any_strides = optional, set(free), any_strides


def _a(name, dtype, shape, align=4, **kw):
    return Arg(name, dtype, shape, align, **kw)


# ----------------------------------------------------------------------------- the table
# Each entry: (case name, entry point, args, workspace: "required" | "optional" | None, invoke(L, lib, t, ws, ws_bytes)).
# t[name] is a DLTensor* (or None); lib is objectdetection_b200._lib (parameter structs).

def _spec(lib):
    return lib.make_anchor_spec((64, 64), [8.0], [1.0], [(4, 4)], [16], 1)   # 16 anchors


def _entries():
    E = []

    def add(name, args, ws, invoke):
        E.append((name, args, ws, invoke))

    add("od_gen_anchors_normalized", [_a("anchors", "f32", (2, 16, 4), 16, free=[0])], None,
        lambda L, lib, t, ws, n: L.od_gen_anchors(ctypes.byref(_spec(lib)), 1, t["anchors"], None))
    add("od_gen_anchors_pixel", [_a("anchors", "f64", (16, 4), 8)], None,
        lambda L, lib, t, ws, n: L.od_gen_anchors(ctypes.byref(_spec(lib)), 0, t["anchors"], None))
    add("od_apply_box_deltas", [_a("boxes", "f32", (2, 3, 4), 16), _a("deltas", "f32", (2, 3, 4), 16),
                                _a("out", "f32", (2, 3, 4), 16)], None,
        lambda L, lib, t, ws, n: L.od_apply_box_deltas(t["boxes"], t["deltas"], t["out"], None))
    add("od_clip_boxes", [_a("boxes", "f32", (2, 3, 4), 16), _a("window", "f32", (2, 4), 16),
                          _a("out", "f32", (2, 3, 4), 16)], None,
        lambda L, lib, t, ws, n: L.od_clip_boxes(t["boxes"], t["window"], t["out"], None))
    add("od_norm_boxes", [_a("boxes", "f32", (2, 3, 4), 4), _a("out", "f32", (2, 3, 4), 16)], None,
        lambda L, lib, t, ws, n: L.od_norm_boxes(t["boxes"], 64, 64, 0, t["out"], None))
    add("od_topk", [_a("scores", "f32", (2, 8), 4, free=[1], any_strides=True), _a("values", "f32", (2, 3), optional=True),
                    _a("indices", "i32", (2, 3))], "required",
        lambda L, lib, t, ws, n: L.od_topk(t["scores"], 3, t["values"], t["indices"], ws, n, None))
    add("od_nms", [_a("boxes", "f32", (2, 5, 4), 16), _a("scores", "f32", (2, 5)), _a("num_valid", "i32", (2,), optional=True),
                   _a("keep_idx", "i32", (2, 3)), _a("num_kept", "i32", (2,), optional=True)], "required",
        lambda L, lib, t, ws, n: L.od_nms(t["boxes"], t["scores"], t["num_valid"], 0.5, 3, t["keep_idx"], t["num_kept"],
                                          ws, n, None))

    def proposal_debug(lib, t):
        return lib.ProposalDebug(*[t["debug." + f] for f, _ in lib.ProposalDebug._fields_])

    def debug_args(K, N):
        return [_a("debug.ix", "i32", (2, K), optional=True), _a("debug.scores", "f32", (2, K), optional=True),
                _a("debug.bbox_delta", "f32", (2, K, 4), 16, optional=True),
                _a("debug.anchors", "f32", (2, K, 4), 16, optional=True),
                _a("debug.anchor_delta", "f32", (2, K, 4), 16, optional=True),
                _a("debug.anchor_delta_clipped", "f32", (2, K, 4), 16, optional=True),
                _a("debug.keep_idx", "i32", (2, N), optional=True), _a("debug.num_kept", "i32", (2,), optional=True)]

    def proposal_params(lib, K, N):
        return lib.ProposalParams((1.0, 1.0, 1.0, 1.0), K, N, 0.7)

    add("od_proposal_forward",
        [_a("rpn_class_probs", "f32", (2, 16, 2)), _a("rpn_bbox", "f32", (2, 16, 4), 16), _a("anchors", "f32", (2, 16, 4), 16),
         _a("proposals", "f32", (2, 4, 4), 16)] + debug_args(8, 4), "required",
        lambda L, lib, t, ws, n: L.od_proposal_forward(
            t["rpn_class_probs"], t["rpn_bbox"], t["anchors"], None, ctypes.byref(proposal_params(lib, 8, 4)), t["proposals"],
            ctypes.byref(proposal_debug(lib, t)), ws, n, None))

    def levels_call(L, lib, t, ws, n):
        logits = (c_void_p * 2)(t["class_logits[0]"], t["class_logits[1]"])
        bbox = (c_void_p * 2)(t["bbox[0]"], t["bbox[1]"])
        return L.od_proposal_forward_levels(logits, bbox, 2, t["anchors"], None, ctypes.byref(proposal_params(lib, 4, 3)),
                                            t["proposals"], ctypes.byref(proposal_debug(lib, t)), ws, n, None)
    add("od_proposal_forward_levels",
        [_a("class_logits[0]", "f32", (2, 2, 2, 2), 8), _a("bbox[0]", "f32", (2, 2, 2, 4), 16),
         _a("class_logits[1]", "f32", (2, 1, 2, 4), 8), _a("bbox[1]", "f32", (2, 1, 2, 8), 16),
         _a("anchors", "f32", (2, 8, 4), 16), _a("proposals", "f32", (2, 3, 4), 16)] + debug_args(4, 3), "required",
        levels_call)

    roi_args = [_a("fmaps[0]", "f32", (2, 4, 4, 8), 16, free=[1, 2]), _a("fmaps[1]", "f32", (2, 2, 2, 8), 16, free=[1, 2]),
                _a("rois", "f32", (2, 3, 4), 16), _a("pooled", "f32", (6, 2, 2, 8), 16),
                _a("roi_level", "i32", (2, 3), optional=True)]

    def fm(t):
        return (c_void_p * 2)(t["fmaps[0]"], t["fmaps[1]"])
    add("od_pyramid_roi_align_forward", roi_args, None,
        lambda L, lib, t, ws, n: L.od_pyramid_roi_align_forward(fm(t), 2, 2, t["rois"], 64, 64, 2, 2, t["pooled"],
                                                                t["roi_level"], None))
    add("od_pyramid_roi_align_forward_ws", roi_args, "optional",
        lambda L, lib, t, ws, n: L.od_pyramid_roi_align_forward_ws(fm(t), 2, 2, t["rois"], 64, 64, 2, 2, t["pooled"],
                                                                   t["roi_level"], ws, n, None))
    add("od_pyramid_roi_align_forward_ordered", roi_args + [_a("order", "i32", (6,), optional=True)], "optional",
        lambda L, lib, t, ws, n: L.od_pyramid_roi_align_forward_ordered(fm(t), 2, 2, t["rois"], 64, 64, 2, 2, t["pooled"],
                                                                        t["roi_level"], t["order"], ws, n, None))
    add("od_roi_processing_order", [_a("rois", "f32", (2, 3, 4), 16), _a("order", "i32", (6,))], None,
        lambda L, lib, t, ws, n: L.od_roi_processing_order(t["rois"], 64, 64, 2, 2, t["order"], None))
    add("od_crop_and_resize", [_a("image", "f32", (2, 4, 4, 8), 16, free=[0, 1, 2]), _a("boxes", "f32", (3, 4), 16),
                               _a("box_ind", "i32", (3,)), _a("out", "f32", (3, 2, 2, 8), 16)], None,
        lambda L, lib, t, ws, n: L.od_crop_and_resize(t["image"], t["boxes"], t["box_ind"], 2, 2, 0.0, t["out"], None))

    def target_call(L, lib, t, ws, n):
        p = lib.TargetParams(4, (0.1, 0.1, 0.2, 0.2), 7, 7, 0, 0)
        dbg = lib.TargetDebug(*[t["debug." + f] for f, _ in lib.TargetDebug._fields_])
        return L.od_detection_target_forward(t["proposals"], t["gt_class_ids"], t["gt_boxes"], t["perm_pos"], t["perm_neg"],
                                             ctypes.byref(p), t["rois"], t["roi_gt_class_ids"], t["roi_gt_box_deltas"],
                                             t["gt_masks"], t["mask_targets"], ctypes.byref(dbg), ws, n, None)
    add("od_detection_target_forward",
        [_a("proposals", "f32", (2, 5, 4), 16), _a("gt_class_ids", "i32", (2, 3)), _a("gt_boxes", "f32", (2, 3, 4), 16),
         _a("perm_pos", "i32", (2, 5)), _a("perm_neg", "i32", (2, 5)), _a("rois", "f32", (2, 4, 4), 16),
         _a("roi_gt_class_ids", "i32", (2, 4)), _a("roi_gt_box_deltas", "f32", (2, 4, 4), 16),
         _a("gt_masks", "f32", (2, 3, 6, 6), free=[2, 3]), _a("mask_targets", "f32", (2, 4, 7, 7)),
         _a("debug.iou", "f32", (2, 5, 3), optional=True), _a("debug.roi_iou_max", "f32", (2, 5), optional=True),
         _a("debug.pos_indices", "i32", (2, 5), optional=True), _a("debug.neg_indices", "i32", (2, 5), optional=True),
         _a("debug.counts", "i32", (2, 6), optional=True), _a("debug.sampled_pos", "i32", (2, 4), optional=True),
         _a("debug.sampled_neg", "i32", (2, 4), optional=True), _a("debug.gt_assignment", "i32", (2, 4), optional=True)],
        "required", target_call)

    def rpn_target_call(L, lib, t, ws, n):
        p = lib.RpnTargetParams(4, (0.1, 0.1, 0.2, 0.2))
        return L.od_rpn_target_forward(t["anchors"], t["gt_boxes"], t["gt_count"], t["perm_pos"], t["perm_neg"],
                                       ctypes.byref(p), t["rpn_target_class"], t["rpn_target_bbox"], t["positive_anchors"],
                                       t["counts"], ws, n, None)
    add("od_rpn_target_forward",
        [_a("anchors", "f64", (6, 4), 8), _a("gt_boxes", "f64", (2, 3, 4), 8, free=[1]), _a("gt_count", "i32", (2,)),
         _a("perm_pos", "i32", (2, 6)), _a("perm_neg", "i32", (2, 6)), _a("rpn_target_class", "i32", (2, 6)),
         _a("rpn_target_bbox", "f64", (2, 4, 4), 8), _a("positive_anchors", "f64", (2, 4, 4), 8),
         _a("counts", "i32", (2, 4))], "required", rpn_target_call)
    add("od_rpn_loss_forward",
        [_a("rpn_target_class", "i32", (2, 6)), _a("rpn_class_logits", "f32", (2, 6, 2), 8),
         _a("rpn_target_bbox", "f32", (2, 3, 4), 16, free=[1]), _a("rpn_pred_box", "f32", (2, 6, 4), 16),
         _a("losses", "f32", (2,)), _a("pred_box_pos", "f32", (5, 4), 16, optional=True, free=[0]),
         _a("num_pos", "i32", (1,), optional=True)], "required",
        lambda L, lib, t, ws, n: L.od_rpn_loss_forward(t["rpn_target_class"], t["rpn_class_logits"], t["rpn_target_bbox"],
                                                       t["rpn_pred_box"], t["losses"], t["pred_box_pos"], t["num_pos"],
                                                       ws, n, None))
    add("od_mrcnn_loss_forward",
        [_a("mrcnn_target_class_ids", "i32", (2, 3)), _a("mrcnn_pred_logits", "f32", (2, 3, 4)),
         _a("batch_active_class_ids", "f32", (2, 4), free=[0]), _a("mrcnn_target_box", "f32", (2, 3, 4), 16),
         _a("mrcnn_pred_box", "f32", (2, 3, 4, 4), 16), _a("losses", "f32", (2,)),
         _a("pred_active", "f32", (2, 3), optional=True)], None,
        lambda L, lib, t, ws, n: L.od_mrcnn_loss_forward(t["mrcnn_target_class_ids"], t["mrcnn_pred_logits"],
                                                         t["batch_active_class_ids"], t["mrcnn_target_box"],
                                                         t["mrcnn_pred_box"], t["losses"], t["pred_active"], None))

    def detection_call(L, lib, t, ws, n):
        p = lib.DetectionParams((0.1, 0.1, 0.2, 0.2), 0.7, 0.3, 4)
        dbg = lib.DetectionDebug(*[t["debug." + f] for f, _ in lib.DetectionDebug._fields_])
        return L.od_detection_forward(t["proposals"], t["mrcnn_class_probs"], t["mrcnn_bbox"], t["window_norm"],
                                      ctypes.byref(p), t["detections"], ctypes.byref(dbg), ws, n, None)
    add("od_detection_forward",
        [_a("proposals", "f32", (2, 5, 4), 16), _a("mrcnn_class_probs", "f32", (2, 5, 3)),
         _a("mrcnn_bbox", "f32", (2, 5, 3, 4), 16), _a("window_norm", "f32", (2, 4), 16), _a("detections", "f32", (2, 4, 6)),
         _a("debug.class_ids", "i32", (2, 5), optional=True), _a("debug.class_scores", "f32", (2, 5), optional=True),
         _a("debug.bbox_delta", "f32", (2, 5, 4), 16, optional=True),
         _a("debug.refined_proposals", "f32", (2, 5, 4), 16, optional=True),
         _a("debug.clipped_proposals", "f32", (2, 5, 4), 16, optional=True),
         _a("debug.keep_mask", "i32", (2, 5), optional=True), _a("debug.nms_keep_mask", "i32", (2, 5), optional=True)],
        "required", detection_call)
    add("od_unmold_detections",
        [_a("detections", "f32", (2, 4, 6)), _a("window_norm", "f32", (2, 4), 16), _a("original_shape", "i32", (2, 2)),
         _a("boxes", "i32", (2, 4, 4)), _a("class_ids", "i32", (2, 4)), _a("scores", "f32", (2, 4)), _a("counts", "i32", (2,))],
        None,
        lambda L, lib, t, ws, n: L.od_unmold_detections(t["detections"], t["window_norm"], t["original_shape"], t["boxes"],
                                                        t["class_ids"], t["scores"], t["counts"], None))

    def frcnn_call(L, lib, t, ws, n):
        p = lib.FrcnnParams()
        p.feat_stride, p.image_h, p.image_w, p.min_box_hw = 16, 64, 64, 16
        p.pre_nms_top_n, p.post_nms_top_n, p.nms_threshold, p.num_anchors = 10, 5, 0.7, 2
        for i, v in enumerate((-8, -8, 23, 23, -16, -16, 31, 31)):
            p.base_anchors[i] = v
        return L.od_frcnn_proposal_forward(t["rpn_box_class_prob"], t["rpn_bbox"], ctypes.byref(p), t["proposals"],
                                           t["num_out"], ws, n, None)
    add("od_frcnn_proposal_forward",
        [_a("rpn_box_class_prob", "f32", (1, 2, 3, 4)), _a("rpn_bbox", "f32", (1, 2, 3, 8)), _a("proposals", "f32", (5, 5)),
         _a("num_out", "i32", (1,))], "required", frcnn_call)
    add("od_roi_pool_forward",
        [_a("feature_map", "f32", (2, 4, 4, 8), 16, free=[0, 1, 2]), _a("proposals", "f32", (3, 5)),
         _a("out", "f32", (3, 7, 7, 8), 16)], None,
        lambda L, lib, t, ws, n: L.od_roi_pool_forward(t["feature_map"], t["proposals"], 64.0, 64.0, t["out"], None))
    return E


ENTRIES = {e[0]: e for e in _entries()}
TENSOR_ENTRY_POINTS = 21   # od_gen_anchors has two baselines, one per mode


def _cases():
    """(case id, entry, mutated arg or None, defect, expected status)."""
    C = []
    for name, args, ws, _ in ENTRIES.values():
        C.append((f"{name}-baseline", name, None, "baseline", ACCEPTED))
        multi = len(args) > 1
        for a in args:
            vec = a.align > 4
            if a.optional:
                C.append((f"{name}-{a.name}-omitted", name, a.name, "null", ACCEPTED))
            else:
                C.append((f"{name}-{a.name}-null", name, a.name, "null", -1))
            C.append((f"{name}-{a.name}-dtype", name, a.name, "dtype", -2))
            C.append((f"{name}-{a.name}-rank+1", name, a.name, "rank+1", -3))
            C.append((f"{name}-{a.name}-rank-1", name, a.name, "rank-1", -3))
            for d in range(len(a.shape)):
                C.append((f"{name}-{a.name}-extent{d}+1", name, a.name, f"extent{d}", ACCEPTED if d in a.free else -3))
            if any(s > 1 for s in a.shape):
                C.append((f"{name}-{a.name}-strided", name, a.name, "strided", ACCEPTED if a.any_strides else -5))
            C.append((f"{name}-{a.name}-offset4", name, a.name, "offset4", -5 if vec else ACCEPTED))
            C.append((f"{name}-{a.name}-device1", name, a.name, "device1", -4 if multi else ACCEPTED))
            C.append((f"{name}-{a.name}-cpu", name, a.name, "cpu", -4))
        if ws == "required":
            C.append((f"{name}-ws-null", name, None, "ws-null", -6))
            C.append((f"{name}-ws-small", name, None, "ws-small", -6))
        elif ws == "optional":
            C.append((f"{name}-ws-null", name, None, "ws-null", ACCEPTED))
            C.append((f"{name}-ws-small", name, None, "ws-small", -6))
    return C


CASES = _cases()


# ----------------------------------------------------------------------------- the child process
def _tensor(arg, defect, keep, base_ptr):
    shape = list(arg.shape)
    if defect == "rank+1":
        shape.append(2)
    elif defect == "rank-1":
        shape.pop()
    elif defect.startswith("extent"):
        shape[int(defect[6:])] += 1
    t = DLTensor()
    t.data = base_ptr
    t.device.device_type, t.device.device_id = (kDLCPU if defect == "cpu" else kDLCUDA), (1 if defect == "device1" else 0)
    t.ndim = len(shape)
    t.dtype.code, t.dtype.bits = WRONG_DTYPE if defect == "dtype" else DTYPES[arg.dtype]
    t.dtype.lanes = 1
    sh = (c_int64 * max(1, len(shape)))(*shape)
    keep.append(sh)
    t.shape = sh
    if defect == "strided":   # every stride doubled: not C-contiguous
        st, acc = [], 1
        for s in reversed(shape):
            st.insert(0, 2 * acc)
            acc *= s
        sa = (c_int64 * len(st))(*st)
        keep.append(sa)
        t.strides = sa
    t.byte_offset = 4 if defect == "offset4" else 0
    keep.append(t)
    return ctypes.cast(ctypes.pointer(t), c_void_p).value


def _worker():
    """Runs every case; refuses to run where a GPU could be visible."""
    if os.environ.get("CUDA_VISIBLE_DEVICES") != "":
        raise SystemExit("refusing to run: CUDA_VISIBLE_DEVICES must be empty")
    sys.path.insert(0, ROOT)
    from objectdetection_b200 import _lib
    import torch
    if torch.cuda.device_count() != 0:
        raise SystemExit("refusing to run: a CUDA device is visible")
    L = _lib.lib()
    out = {}
    for cid, entry, target, defect, _ in CASES:
        name, args, _, invoke = ENTRIES[entry]
        keep, t = [], {}
        for i, a in enumerate(args):
            ptr = 0x10000000 * (i + 1)   # fake, 256-byte aligned, never dereferenced
            if a.name == target and defect == "null":
                t[a.name] = None
            else:
                t[a.name] = _tensor(a, defect if a.name == target else "baseline", keep, ptr)
        ws, n = 0x7F0000000000, WS_BYTES
        if defect == "ws-null":
            ws = None
        elif defect == "ws-small":
            n = 1
        before = L.od_launch_count()
        status = invoke(L, _lib, t, ws, n)
        out[cid] = [status, L.od_last_error_detail().decode(errors="replace"), L.od_launch_count() != before]
    json.dump(out, sys.stdout)


@pytest.fixture(scope="module")
def results():
    """All cases, run once in a child process that cannot see a GPU (the environment is set here, not by the caller)."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    flags = ["-s"] if sys.flags.no_user_site else []
    r = subprocess.run([sys.executable, *flags, os.path.abspath(__file__), "--worker"], env=env, cwd=ROOT,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    return json.loads(r.stdout)


def test_table_covers_every_tensor_entry_point():
    from objectdetection_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "odhead.h")).read()
    takes_tensors = {n for n in _lib.SIGNATURES if re.search(r"\b%s\s*\([^;]*DLTensor" % n, hdr)}
    covered = {e.split("_normalized")[0].split("_pixel")[0] for e in ENTRIES}
    assert covered == takes_tensors
    assert len(takes_tensors) == TENSOR_ENTRY_POINTS


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_validation_status(results, case):
    cid, _, target, defect, expected = case
    status, detail, launched = results[cid]
    assert status == expected, f"{cid}: status {status}, expected {expected} ({detail})"
    if expected != ACCEPTED:
        assert not launched, f"{cid}: refused with {status} after a launch"


@pytest.mark.parametrize("case", [c for c in CASES if c[4] != ACCEPTED and c[2]], ids=[c[0] for c in CASES if c[4] != ACCEPTED and c[2]])
def test_validation_detail_names_argument(results, case):
    cid, _, target, defect, expected = case
    status, detail, _ = results[cid]

    def names(arg):
        return re.search(r"(?<![\w.])" + re.escape(re.sub(r"\[\d\]", "[l]", arg)) + r"(?!\w)", detail)
    if defect.startswith("extent"):
        # an extent shared by several arguments is reported on whichever of them is checked against it
        ok = any(names(a.name) for a in ENTRIES[case[1]][1]) and re.search(r"extent \d is \d+, expected", detail)
    elif defect == "device1":
        # a wrong device on the call's first tensor makes it the call's device; the next tensor is reported against it
        ok = names(target) or "expected cuda:1" in detail
    else:
        ok = names(target)
    assert ok, f"{cid}: detail {detail!r}"


if __name__ == "__main__" and sys.argv[1:] == ["--worker"]:
    _worker()
