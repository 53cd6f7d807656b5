"""Argument validation of the bfloat16 head outputs, CPU only.

od_proposal_forward_levels, od_proposal_forward, od_detection_forward, od_rpn_loss_forward and od_mrcnn_loss_forward
take the tensors a network head produces (RPN logits and deltas, classifier probabilities and boxes, the loss inputs) in
float32 or bfloat16, each argument on its own. A bfloat16 tensor must be aligned to the kernel's load: 2 bytes for a
scalar, 4 for a (bg, fg) logit pair, 8 for a 4-value box row. float16 is still refused, and so is bfloat16 for every
other argument. The calls run in one child process that sees no GPU, like test_abi_validation.py, whose table and
tensor layout they reuse: a call that passes validation returns OD_ERR_CUDA (-7) at its first CUDA call."""
import ctypes
import json
import os
import re
import subprocess
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from test_abi_validation import ACCEPTED, DTYPES, ENTRIES, ROOT, WS_BYTES, DLTensor, kDLCUDA  # noqa: E402

BF16, F16 = (4, 16), (2, 16)
ERR_DTYPE, ERR_LAYOUT = -2, -5

# (entry point, argument group, bf16 alignment): a group is the argument, or every level of a level list
BF16_ARGS = [
    ("od_proposal_forward_levels", ("class_logits[0]", "class_logits[1]"), 4),
    ("od_proposal_forward_levels", ("bbox[0]", "bbox[1]"), 8),
    ("od_proposal_forward", ("rpn_bbox",), 8),
    ("od_detection_forward", ("mrcnn_class_probs",), 2),
    ("od_detection_forward", ("mrcnn_bbox",), 8),
    ("od_rpn_loss_forward", ("rpn_class_logits",), 4),
    ("od_rpn_loss_forward", ("rpn_pred_box",), 8),
    ("od_mrcnn_loss_forward", ("mrcnn_pred_logits",), 2),
    ("od_mrcnn_loss_forward", ("mrcnn_pred_box",), 8),
]

# arguments that stay float32 in every entry point above
F32_ONLY = {
    "od_proposal_forward_levels": ["anchors", "proposals", "debug.scores", "debug.bbox_delta", "debug.anchor_delta_clipped"],
    "od_proposal_forward": ["rpn_class_probs", "anchors", "proposals", "debug.bbox_delta", "debug.anchors"],
    "od_detection_forward": ["proposals", "window_norm", "detections", "debug.class_scores", "debug.bbox_delta",
                             "debug.refined_proposals"],
    "od_rpn_loss_forward": ["rpn_target_bbox", "losses", "pred_box_pos"],
    "od_mrcnn_loss_forward": ["batch_active_class_ids", "mrcnn_target_box", "losses", "pred_active"],
}


def _cases():
    """(case id, entry, {argument: (dtype, byte_offset)}, expected status, argument the detail names or None)."""
    C = []
    for entry, group, align in BF16_ARGS:
        tag = group[0].split("[")[0]
        C.append((f"{entry}-{tag}-bf16", entry, {a: (BF16, 0) for a in group}, ACCEPTED, None))
        C.append((f"{entry}-{tag}-bf16-misaligned", entry, {**{a: (BF16, 0) for a in group}, group[-1]: (BF16, align // 2)},
                  ERR_LAYOUT, group[-1]))
        C.append((f"{entry}-{tag}-f16", entry, {a: (F16, 0) for a in group}, ERR_DTYPE, group[0]))
        if len(group) > 1:
            C.append((f"{entry}-{tag}-mixed-bf16-first", entry, {group[0]: (BF16, 0)}, ERR_DTYPE, group[1]))
            C.append((f"{entry}-{tag}-mixed-f32-first", entry, {group[1]: (BF16, 0)}, ERR_DTYPE, group[1]))
    # both bf16-capable arguments of an entry point in bf16 together (each alone is covered above)
    for entry in ("od_proposal_forward_levels", "od_detection_forward", "od_rpn_loss_forward", "od_mrcnn_loss_forward"):
        over = {a: (BF16, 0) for e, group, _ in BF16_ARGS if e == entry for a in group}
        C.append((f"{entry}-all-bf16", entry, over, ACCEPTED, None))
        for name in F32_ONLY[entry]:
            C.append((f"{entry}-all-bf16-{name}-f16", entry, {**over, name: (F16, 0)}, ERR_DTYPE, name))
    for entry, names in F32_ONLY.items():
        for name in names:
            C.append((f"{entry}-{name}-bf16", entry, {name: (BF16, 0)}, ERR_DTYPE, name))
    return C


CASES = _cases()


def _tensor(arg, over, keep, ptr):
    dtype, offset = over if over else (DTYPES[arg.dtype], 0)
    t = DLTensor()
    t.data = ptr
    t.device.device_type, t.device.device_id = kDLCUDA, 0
    t.ndim = len(arg.shape)
    t.dtype.code, t.dtype.bits = dtype
    t.dtype.lanes = 1
    sh = (ctypes.c_int64 * len(arg.shape))(*arg.shape)
    t.shape = sh
    t.byte_offset = offset
    keep.extend([sh, t])
    return ctypes.cast(ctypes.pointer(t), ctypes.c_void_p).value


def _worker():
    if os.environ.get("CUDA_VISIBLE_DEVICES") != "":
        raise SystemExit("refusing to run: CUDA_VISIBLE_DEVICES must be empty")
    sys.path.insert(0, ROOT)
    from objectdetection_b200 import _lib
    import torch
    if torch.cuda.device_count() != 0:
        raise SystemExit("refusing to run: a CUDA device is visible")
    L = _lib.lib()
    out = {}
    for cid, entry, over, _, _ in CASES:
        _, args, _, invoke = ENTRIES[entry]
        missing = set(over) - {a.name for a in args}
        assert not missing, (cid, missing)
        keep = []
        t = {a.name: _tensor(a, over.get(a.name), keep, 0x10000000 * (i + 1)) for i, a in enumerate(args)}
        before = L.od_launch_count()
        status = invoke(L, _lib, t, 0x7F0000000000, WS_BYTES)
        out[cid] = [status, L.od_last_error_detail().decode(errors="replace"), L.od_launch_count() != before]
    json.dump(out, sys.stdout)


@pytest.fixture(scope="module")
def results():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    flags = ["-s"] if sys.flags.no_user_site else []
    r = subprocess.run([sys.executable, *flags, os.path.abspath(__file__), "--worker"], env=env, cwd=ROOT,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    return json.loads(r.stdout)


def test_table_names_existing_arguments():
    for entry, group, _ in BF16_ARGS:
        assert {a.name for a in ENTRIES[entry][1]} >= set(group) | set(F32_ONLY[entry])


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_bf16_head_validation(results, case):
    cid, _, _, expected, name = case
    status, detail, launched = results[cid]
    assert status == expected, f"{cid}: status {status}, expected {expected} ({detail})"
    if expected != ACCEPTED:
        assert not launched, f"{cid}: refused with {status} after a launch"
        want = re.sub(r"\[\d\]", "[l]", name)   # the levels are reported as class_logits[l] / bbox[l]
        assert re.search(r"(?<![\w.])" + re.escape(want) + r"(?!\w)", detail), f"{cid}: detail {detail!r} does not name {want}"
    if "mixed" in cid:
        assert "level 1" in detail, f"{cid}: detail {detail!r} does not name the level"


if __name__ == "__main__" and sys.argv[1:] == ["--worker"]:
    _worker()
