"""Mask targets from uint8 and bool GT masks (mask_target_kernel<unsigned char>), the dtypes mask datasets store masks
in. A byte widens to fp32 exactly and everything after the load is the fp32 path, so every case compares the targets,
bit for bit, with those of the float32 call on the widened masks and with the oracle on the widened array. Outputs are
pre-filled with a sentinel that must be overwritten everywhere.

The cases: both layouts, mini and full-size masks (1024 x 1024), non-square masks and targets, targets of 1 x 1, exact
0.5 ties, uint8 values across 0..255, GT padding at the start, in the middle and interleaved, near-degenerate GT boxes,
R at the 4096 cap of the mask targets and G at the 8192 cap of GT boxes. A kernel trace shows which kernel served a
dtype, and that BuildDetectionTargets hands bool and uint8 masks, CUDA tensors or host arrays, to the library without a
conversion kernel."""
import ctypes
import functools
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
from test_gpu_dispatch import _many_gt_inputs, assert_launched  # noqa: E402
from test_gpu_unpinned_outputs import _blob_masks, check_masks_against_f64, mask_case  # noqa: E402

import oracle  # noqa: E402
from objectdetection_b200.config import config as Conf  # noqa: E402

torch = pytest.importorskip("torch")
f32 = np.float32
SENTINEL = 0x7FBADBAD


@pytest.fixture(scope="module")
def _cuda():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (there is no CPU path)")


# ------------------------------------------------------------------ inputs
def _denormal_gt():
    """GT boxes one denormal high (or wide): a proposal equal to one (IoU 1) and one twice as high (IoU exactly 0.5, a
    positive) whose box in the GT frame reaches y = 2, so that with mini masks half its rows sample outside the mask and
    take the extrapolation value. Zero-height and zero-width GT rows of a valid class sit beside them; their IoU is 0
    with every proposal, so none is assigned, and they stay out of the way of the compacted GT indices."""
    rs = np.random.RandomState(7)
    d = np.nextafter(f32(0), f32(1))                          # the smallest denormal
    gt = np.array([[[0, 0, d, 1], [0.5, 0.2, 0.5, 0.8], [0, 0, 1, d], [0.2, 0.4, 0.8, 0.4], [0.3, 0.3, 0.6, 0.7]]], f32)
    cls = np.array([[3, 4, 5, 6, 7]], np.int32)
    props = np.zeros((1, 64, 4), f32)
    props[0, :4] = [[0, 0, d, 1], [0, 0, 2 * d, 1], [0, 0, 1, d], [0, 0, 1, 2 * d]]
    props[0, 4] = gt[0, 4]
    props[0, 5:50] = _synth.random_boxes(rs, 45) * f32(0.2) + f32(0.75)
    pp = pn = np.arange(64, dtype=np.int32)[None]
    masks = (_blob_masks(rs, 1, 20, 16, 5) > 0).astype(np.uint8)
    masks[..., :3] = 1                                        # the thin boxes' masks: ones, so extrapolated rows show
    return (28, 28), 200, props, cls, gt, pp, pn, masks


@functools.lru_cache(maxsize=None)
def inputs(name):
    """(mask_shape, R, props, cls, gt, pp, pn, masks [B,Mh,Mw,G] uint8) of one named case."""
    if name == "nonsquare_48x40_to_28x14":
        rs = np.random.RandomState(13)
        props, cls, gt, pp, pn = _synth.target_inputs(rs, 3, 600, 20, n_pad=100)
        return (28, 14), 200, props, cls, gt, pp, pn, (_blob_masks(rs, 3, 48, 40, 20) > 0).astype(np.uint8)
    if name == "u8_values":
        # every value 0..255 (odd sums at half-pixel taps give exact .5 ties), with rows of the extremes 0 and 255
        rs = np.random.RandomState(255)
        props, cls, gt, pp, pn = _synth.target_inputs(rs, 2, 600, 20, n_pad=100)
        masks = rs.randint(0, 256, (2, 32, 24, 20))
        masks[:, :4] = 255
        masks[:, -4:] = 0
        return (28, 28), 200, props, cls, gt, pp, pn, masks.astype(np.uint8)
    if name == "gt_8192":
        rs = np.random.RandomState(8192)
        props, cls, gt, pp, pn = _many_gt_inputs(rs, 2, 2000, 8192)
        return (28, 28), 200, props, cls, gt, pp, pn, (_blob_masks(rs, 2, 6, 5, 8192) > 0).astype(np.uint8)
    if name == "denormal_gt":
        return _denormal_gt()
    shape, R, props, cls, gt, pp, pn, masks = mask_case(name)
    assert set(np.unique(masks)) <= {0.0, 1.0}, name
    return shape, R, props, cls, gt, pp, pn, masks.astype(np.uint8)


# mini masks (56 x 40, 28 x 36, 20 x 24 ...) and full-size 1024 x 1024 masks; each runs with use_mini_mask on and off
CASES = ["pad_start", "pad_middle", "pad_interleaved", "nonsquare_48x40_to_28x14", "shape_1x1", "exact_tie",
         "u8_values", "thin_gt", "denormal_gt", "full_image_1024", "rois_4096", "gt_8192"]


def byte_masks(masks, dtype):
    return masks.astype(bool) if dtype == "bool" else masks


@functools.lru_cache(maxsize=None)
def oracle_rois(name):
    shape, R, props, cls, gt, pp, pn, _ = inputs(name)
    return [oracle.detection_targets(props[b], cls[b], gt[b], pp[b], pn[b], R, Conf.BBOX_STD_DEV)
            for b in range(props.shape[0])]


# ------------------------------------------------------------------ device calls
def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    torch.cuda.synchronize()
    return t.detach().cpu().numpy()


def _targets(shape, R, mini, props, cls, gt, pp, pn, masks, hwg):
    """od_detection_target_forward on masks [B,Mh,Mw,G] of any dtype, passed as [B,Mh,Mw,G] (hwg) or [B,G,Mh,Mw], with
    mask_targets pre-filled with SENTINEL. Returns (rois, mask_targets, counts, gt_assignment) on the host."""
    from objectdetection_b200 import _lib
    B, N = props.shape[:2]
    G = cls.shape[1]
    if not hwg:
        masks = masks.transpose(0, 3, 1, 2)
    t = {k: cu(v) for k, v in dict(props=props, cls=cls, gt=gt, pp=pp, pn=pn, masks=masks).items()}
    rois = torch.empty((B, R, 4), dtype=torch.float32, device="cuda")
    rcls = torch.empty((B, R), dtype=torch.int32, device="cuda")
    deltas = torch.empty((B, R, 4), dtype=torch.float32, device="cuda")
    targets = torch.full((B, R) + tuple(shape), SENTINEL, dtype=torch.int32, device="cuda").view(torch.float32)
    counts = torch.empty((B, 6), dtype=torch.int32, device="cuda")
    assign = torch.empty((B, R), dtype=torch.int32, device="cuda")
    params = _lib.TargetParams(R, (ctypes.c_float * 4)(*Conf.BBOX_STD_DEV), shape[0], shape[1], 1 if mini else 0,
                               1 if hwg else 0)
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


def assert_bits(got, want, what):
    assert got.shape == want.shape, (what, got.shape, want.shape)
    bad = got.view(np.uint32) != want.view(np.uint32)
    assert not bad.any(), (what, int(bad.sum()), np.argwhere(bad)[:5].tolist())


# ------------------------------------------------------------------ byte masks == float32 masks
@pytest.mark.gpu
@pytest.mark.parametrize("mini", [True, False], ids=["mini", "full"])
@pytest.mark.parametrize("hwg", [True, False], ids=["hwg", "ghw"])
@pytest.mark.parametrize("dtype", ["uint8", "bool"])
@pytest.mark.parametrize("case", CASES)
def test_byte_masks_equal_float32_masks(_cuda, case, dtype, hwg, mini):
    shape, R, props, cls, gt, pp, pn, masks = inputs(case)
    byte = byte_masks(masks, dtype)
    wide = byte.astype(f32)
    rois, got, counts, _ = _targets(shape, R, mini, props, cls, gt, pp, pn, byte, hwg)
    assert not (got.view(np.uint32) == SENTINEL).any(), "a mask_targets word was not written"
    rois32, want32, counts32, _ = _targets(shape, R, mini, props, cls, gt, pp, pn, wide, hwg)
    assert_bits(rois, rois32, "rois")
    assert np.array_equal(counts, counts32)
    assert_bits(got, want32, "mask_targets vs the float32 call")
    n_pos = counts[:, 4]
    for b, (w_rois, _, _, wd) in enumerate(oracle_rois(case)):
        assert_bits(rois[b], w_rois, f"rois[{b}] vs the oracle")
        want = oracle.mask_targets(w_rois, cls[b], gt[b], wide[b], wd, shape, mini)
        assert_bits(got[b], want, f"mask_targets[{b}] vs the oracle")
    assert n_pos.sum() > 0 and got.any()
    if case == "exact_tie":
        assert n_pos[0] >= 1 and np.array_equal(got[0, 0], np.tile([0, 0, 1, 0, 0], (5, 1)))
    if case == "u8_values" and dtype == "uint8":
        assert got.max() == 255 and np.any((got > 1) & (got < 255))
    if case == "denormal_gt":
        assert n_pos[0] == 5, n_pos                        # the four thin proposals and the copy of GT row 4
        tall = [r for r in range(5) if np.array_equal(rois[0, r].view(np.uint32), props[0, 1].view(np.uint32))]
        assert len(tall) == 1
        if mini:             # box y 0..2 in the GT frame: rows past the mask are 0 (the last column may round past it)
            assert got[0, tall[0], :14].any(1).all() and not got[0, tall[0], 14:].any()
    if case == "rois_4096":
        assert (n_pos == 1351).all(), n_pos
    if case == "gt_8192":
        assert max(int(a) for b in range(2) for a in oracle_rois(case)[b][3]["gt_assignment"][:n_pos[b]]) > 4096


@pytest.mark.gpu
@pytest.mark.parametrize("hwg", [True, False], ids=["hwg", "ghw"])
def test_bool_masks_against_f64(_cuda, hwg):
    """The float64 restatement of tests/_f64_refs.py on bool masks: exact on every pixel it can decide."""
    shape, R, props, cls, gt, pp, pn, masks = inputs("pad_interleaved")
    rois, got, counts, assign = _targets(shape, R, True, props, cls, gt, pp, pn, masks.astype(bool), hwg)
    check_masks_against_f64(shape, True, props, cls, gt, masks.astype(f32), rois, counts[:, 4], assign, got)


# ------------------------------------------------------------------ BuildDetectionTargets
def _conf():
    class C(Conf):
        USE_MINI_MASK = True
        MASK_SHAPE = (28, 14)
    return C()


def _layer_inputs():
    _, _, props, cls, gt, pp, pn, masks = inputs("nonsquare_48x40_to_28x14")
    return [cu(a) for a in (props, cls, gt, pp, pn)], masks


def _layer(conf, args, m, b=None):
    from objectdetection_b200 import BuildDetectionTargets
    P, C, Gb, PP, PN = args if b is None else [a[b] for a in args]
    return BuildDetectionTargets(conf, P, C, Gb, perm_pos=PP, perm_neg=PN, gt_masks=m).get_target_masks()


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["uint8", "bool"])
@pytest.mark.parametrize("where", ["cuda", "host"])
def test_build_detection_targets_byte_masks(_cuda, where, dtype):
    """A bool or uint8 CUDA tensor or host array gives the targets of the float32 masks, batched and per image."""
    conf = _conf()
    args, masks = _layer_inputs()
    byte = byte_masks(masks, dtype)
    if where == "cuda":
        byte = cu(byte)
    assert_bits(host(_layer(conf, args, byte)), host(_layer(conf, args, cu(masks.astype(f32)))), f"{where} {dtype} masks")
    assert_bits(host(_layer(conf, args, byte[1], 1)), host(_layer(conf, args, cu(masks[1].astype(f32)), 1)),
                f"{where} {dtype} masks, one image")


# ------------------------------------------------------------------ which kernels ran
# BuildDetectionTargets on CUDA tensors and host arrays of each mask dtype. A bool or uint8 mask must reach the library
# without a conversion kernel, so each traced call sits between two fill_ kernels of a probe tensor: the trace must show
# both (its window caught the start and the end of the call) and nothing else outside the library. float16 masks, for
# contrast, are converted to float32 on the device first.
TRACES = ["cuda-uint8", "cuda-bool", "cuda-float32", "cuda-float16", "host-uint8", "host-bool"]
PROBE = "FillFunctor"


def _trace_worker():
    """Traced in a process of its own: in a process that has run many other GPU tests, a profiler session has come back
    without part of its device activity (see test_gpu_roi_align_bf16.py)."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    conf = _conf()
    args, masks = _layer_inputs()
    probe = torch.zeros(1, device="cuda")
    srcs = {"cuda-uint8": cu(masks), "cuda-bool": cu(masks.astype(bool)), "cuda-float32": cu(masks.astype(f32)),
            "cuda-float16": cu(masks.astype(np.float16)), "host-uint8": masks, "host-bool": masks.astype(bool)}
    out = {}
    for name in TRACES:
        _layer(conf, args, srcs[name])                      # workspace outside the window
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA], acc_events=True) as prof:
            probe.fill_(1.0)
            _layer(conf, args, srcs[name])
            probe.fill_(2.0)
            torch.cuda.synchronize()
        out[name] = [e.name for e in prof.events() if e.device_type == DeviceType.CUDA
                     and not e.name.startswith(("Memcpy", "Memset"))]
    json.dump(out, sys.stdout)


@pytest.fixture(scope="module")
def traces(_cuda):
    flags = ["-s"] if sys.flags.no_user_site else []
    r = subprocess.run([sys.executable, *flags, os.path.abspath(__file__), "--trace"], cwd=ROOT, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    return json.loads(r.stdout)


@pytest.mark.gpu
@pytest.mark.parametrize("name", TRACES)
def test_kernel_trace(traces, name):
    names = traces[name]
    probes = [n for n in names if PROBE in n]
    assert len(probes) == 2, f"{name}: the trace does not hold both probe kernels: {sorted(set(names))}"
    outside = sorted({n for n in names if "od::" not in n and PROBE not in n})
    if name.endswith(("uint8", "bool")):
        assert_launched(names, must=["od::mask_target_kernel<unsigned char>("], must_not=["od::mask_target_kernel("])
        assert not outside, f"{name}: kernels outside the library ran: {outside}"
    else:
        assert_launched(names, must=["od::mask_target_kernel("], must_not=["od::mask_target_kernel<"])
        if name == "cuda-float16":
            assert outside, f"{name}: no conversion kernel in the trace"
        else:
            assert not outside, f"{name}: kernels outside the library ran: {outside}"


if __name__ == "__main__" and sys.argv[1:] == ["--trace"]:
    _trace_worker()
