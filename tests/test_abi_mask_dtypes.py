"""Argument validation of the byte GT masks of od_detection_target_forward, CPU only.

gt_masks may be float32, uint8 (kDLUInt, 8 bits) or bool (kDLBool, 8 bits), in either layout ([B,G,Mh,Mw] or, with
mask_layout_hwg, [B,Mh,Mw,G]). A byte mask is read one byte at a time, so it needs no alignment; float32 keeps its 4
bytes. Every other dtype is refused and named, and mask_targets stays float32. The calls run in one child process that
sees no GPU, like test_abi_validation.py, whose table and tensor layout they reuse: a call that passes validation
returns OD_ERR_CUDA (-7) at its first CUDA call."""
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

ENTRY = "od_detection_target_forward"
U8, BOOL = (1, 8), (6, 8)
F32 = DTYPES["f32"]
REFUSED = {"f16": (2, 16), "bf16": (4, 16), "i8": (0, 8), "f64": (2, 64), "i16": (0, 16), "u16": (1, 16),
           "bool16": (6, 16)}
ERR_DTYPE, ERR_LAYOUT = -2, -5
HWG_SHAPE = (2, 6, 6, 3)          # the [B,Mh,Mw,G] form of the table's [B,G,Mh,Mw] = (2, 3, 6, 6) gt_masks


def _cases():
    """(case id, layout_hwg, {argument: (dtype, byte_offset)}, expected status, argument the detail names or None)."""
    C = []
    for hwg in (False, True):
        lay = "hwg" if hwg else "ghw"
        for tag, dt in (("u8", U8), ("bool", BOOL)):
            C.append((f"{lay}-{tag}", hwg, {"gt_masks": (dt, 0)}, ACCEPTED, None))
            C.append((f"{lay}-{tag}-offset1", hwg, {"gt_masks": (dt, 1)}, ACCEPTED, None))
            C.append((f"{lay}-{tag}-targets-u8", hwg, {"gt_masks": (dt, 0), "mask_targets": (U8, 0)}, ERR_DTYPE,
                      "mask_targets"))
        C.append((f"{lay}-f32-offset2", hwg, {"gt_masks": (F32, 2)}, ERR_LAYOUT, "gt_masks"))
        C.append((f"{lay}-f32-targets-u8", hwg, {"mask_targets": (U8, 0)}, ERR_DTYPE, "mask_targets"))
        C.append((f"{lay}-f32-targets-bool", hwg, {"mask_targets": (BOOL, 0)}, ERR_DTYPE, "mask_targets"))
        for tag, dt in REFUSED.items():
            C.append((f"{lay}-{tag}", hwg, {"gt_masks": (dt, 0)}, ERR_DTYPE, "gt_masks"))
    return C


CASES = _cases()


def _tensor(arg, shape, over, keep, ptr):
    dtype, offset = over if over else (DTYPES[arg.dtype], 0)
    t = DLTensor()
    t.data = ptr
    t.device.device_type, t.device.device_id = kDLCUDA, 0
    t.ndim = len(shape)
    t.dtype.code, t.dtype.bits = dtype
    t.dtype.lanes = 1
    sh = (ctypes.c_int64 * len(shape))(*shape)
    t.shape = sh
    t.byte_offset = offset
    keep.extend([sh, t])
    return ctypes.cast(ctypes.pointer(t), ctypes.c_void_p).value


def _hwg_call(L, lib, t, ws, n):
    """The table's call with mask_layout_hwg = 1."""
    p = lib.TargetParams(4, (0.1, 0.1, 0.2, 0.2), 7, 7, 0, 1)
    dbg = lib.TargetDebug(*[t["debug." + f] for f, _ in lib.TargetDebug._fields_])
    return L.od_detection_target_forward(t["proposals"], t["gt_class_ids"], t["gt_boxes"], t["perm_pos"], t["perm_neg"],
                                         ctypes.byref(p), t["rois"], t["roi_gt_class_ids"], t["roi_gt_box_deltas"],
                                         t["gt_masks"], t["mask_targets"], ctypes.byref(dbg), ws, n, None)


def _worker():
    if os.environ.get("CUDA_VISIBLE_DEVICES") != "":
        raise SystemExit("refusing to run: CUDA_VISIBLE_DEVICES must be empty")
    sys.path.insert(0, ROOT)
    from objectdetection_b200 import _lib
    import torch
    if torch.cuda.device_count() != 0:
        raise SystemExit("refusing to run: a CUDA device is visible")
    L = _lib.lib()
    _, args, _, table_call = ENTRIES[ENTRY]
    out = {}
    for cid, hwg, over, _, _ in CASES:
        keep = []
        t = {a.name: _tensor(a, HWG_SHAPE if hwg and a.name == "gt_masks" else a.shape, over.get(a.name), keep,
                             0x10000000 * (i + 1))
             for i, a in enumerate(args)}
        before = L.od_launch_count()
        status = (_hwg_call if hwg else table_call)(L, _lib, t, 0x7F0000000000, WS_BYTES)
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


def test_table_has_the_mask_arguments():
    args = {a.name: a for a in ENTRIES[ENTRY][1]}
    assert args["gt_masks"].dtype == "f32" and args["gt_masks"].shape == (2, 3, 6, 6)
    assert args["mask_targets"].dtype == "f32"


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_mask_dtype_validation(results, case):
    cid, _, _, expected, name = case
    status, detail, launched = results[cid]
    assert status == expected, f"{cid}: status {status}, expected {expected} ({detail})"
    if expected != ACCEPTED:
        assert not launched, f"{cid}: refused with {status} after a launch"
        assert re.search(r"(?<![\w.])" + re.escape(name) + r"(?!\w)", detail), f"{cid}: detail {detail!r} does not name {name}"


if __name__ == "__main__" and sys.argv[1:] == ["--worker"]:
    _worker()
