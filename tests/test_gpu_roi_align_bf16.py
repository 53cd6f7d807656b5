"""bfloat16 feature maps and pooled output of PyramidROIAlign and crop_and_resize.

The blend is fp32 in the reference's order whatever the dtypes: bf16 map values are widened exactly, so a pooled fp32
result from bf16 maps is bit-identical to the fp32 path (and the CPU oracle) on the widened maps, and a bf16 result is
the round-to-nearest-even of that fp32 value (torch's float32 -> bfloat16 conversion; NaN stays NaN). Each of the three
new (maps, pooled) dtype pairs is checked against both, on the shapes and edges test_gpu_parity.py covers for fp32.

The refusal tests at the end need no GPU: they run in a child process that sees none, like test_abi_validation.py."""
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path[:0] = [HERE, ROOT]                  # ROOT: oracle, also in the refusal tests' child process
import _synth  # noqa: E402

import oracle  # noqa: E402
from test_abi_validation import ACCEPTED, DLTensor, kDLCUDA  # noqa: E402
from test_gpu_dispatch import assert_launched  # noqa: E402
from test_gpu_parity import assert_bits, cu, host  # noqa: E402

torch = pytest.importorskip("torch")
f32 = np.float32
gpu = pytest.mark.gpu
F32, BF16 = torch.float32, torch.bfloat16
COMBOS = [(BF16, F32), (F32, BF16), (BF16, BF16)]          # (maps, pooled); fp32 -> fp32 is test_gpu_parity.py's
IDS = ["bf16-f32", "f32-bf16", "bf16-bf16"]


@pytest.fixture(scope="module")
def _cuda():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (there is no CPU path)")


def bf16_values(a):
    """The bf16 value nearest to each element, as fp32 (the maps both paths are fed)."""
    return torch.from_numpy(np.ascontiguousarray(a, f32)).to(BF16).float().numpy()


def rounded(a, dt):
    return bf16_values(a) if dt == BF16 else np.asarray(a, f32)


def got_f32(t, dt):
    assert t.dtype == dt, (t.dtype, dt)
    return host(t.float())


def maps_as(fmaps32, dt):
    return [cu(f).to(dt) for f in fmaps32]


def _pyramid(fmaps32, props, pool, combos=COMBOS, **kw):
    """fmaps32 hold bf16 values. Every combo against the oracle and the fp32 CUDA path, both rounded to the pooled
    dtype."""
    from objectdetection_b200.maskrcnn import pyramid_roi_align
    want, _ = oracle.pyramid_roi_align(fmaps32, props, 1024, 1024, pool[0], pool[1])
    pr = cu(props)
    ref = host(pyramid_roi_align(maps_as(fmaps32, F32), pr, [1024, 1024], pool, **kw))
    assert_bits(ref, want, f"fp32 path {pool}")
    for md, od in combos:
        got = got_f32(pyramid_roi_align(maps_as(fmaps32, md), pr, [1024, 1024], pool, out_dtype=od, **kw), od)
        assert_bits(got, rounded(want, od), f"{md} -> {od} {pool} vs oracle")
        assert_bits(got, rounded(ref, od), f"{md} -> {od} {pool} vs fp32 path")


def _counters_zeroed():
    from objectdetection_b200 import _lib
    torch.cuda.synchronize()
    return all(int(w[:256].count_nonzero()) == 0 for w in _lib._zero_ws.values())


# ------------------------------------------------------------------ parity
@gpu
@pytest.mark.parametrize("pool", [[7, 7], [14, 14]])
def test_bf16_debug_recipe(_cuda, pool):
    """maskrcnn.py:327-345 recipe (seed 255, P2..P5 of 2 images, 2 x 1000 uniform proposals) at bf16 precision."""
    np.random.seed(255)
    fmaps = [bf16_values(np.random.random((2, s, s, 256))) for s in (256, 128, 64, 32)]
    props = np.array(np.random.random((2, 1000, 4)), dtype="float32")
    _pyramid(fmaps, props, pool)


@gpu
@pytest.mark.parametrize("pool", [[7, 7], [14, 14], [1, 1], [3, 5], [16, 16], [5, 14], [14, 2]])
def test_bf16_edge_case_rois(_cuda, pool):
    """Up-/down-sampled, thin, flipped, NaN, zero-area, outside and whole-image ROIs: the flat per-bin path inside
    crop_rows_kernel and both crop_bins_kernel tables; the ticket counters are left zeroed."""
    rs = np.random.RandomState(4321 + pool[0])
    fmaps = [bf16_values(rs.random_sample((2, s, s, 256))) for s in (64, 32, 16, 8)]
    props = _synth.rois_with_edge_cases(rs, 2, 160)
    _pyramid(fmaps, props, pool)
    assert _counters_zeroed()


@gpu
@pytest.mark.parametrize("pool,n", [([14, 14], 700), ([7, 7], 700), ([14, 14], 4500)])
def test_bf16_processing_order(_cuda, pool, n):
    """>= 512 ROIs: the order pre-pass feeds both kernels; 4500 ROIs per image exceed it (index order)."""
    rs = np.random.RandomState(77 + n + pool[0])
    fmaps = [bf16_values(rs.random_sample((2, s, s, 256))) for s in (64, 32, 16, 8)]
    props = _synth.rois_log_uniform(rs, 2, n, lo=4, hi=900)
    props[0, 3] = [np.nan, 0.1, 0.5, 0.6]
    props[0, 5] = [0.9, 0.1, 0.2, 0.8]
    props[0, 7] = [1.5, 1.5, 2.0, 2.0]
    props[1, n - 50:] = 0
    _pyramid(fmaps, props, pool)


@gpu
@pytest.mark.parametrize("pool", [[14, 14], [7, 7]])
def test_bf16_caller_supplied_and_corrupted_order(_cuda, pool):
    """A caller-supplied order gives the same bits; a corrupted one leaves the rows of skipped ROIs untouched."""
    from objectdetection_b200.maskrcnn import pyramid_roi_align, roi_processing_order
    rs = np.random.RandomState(5 + pool[0])
    fmaps = [bf16_values(rs.random_sample((2, s, s, 256))) for s in (64, 32, 16, 8)]
    props = _synth.rois_log_uniform(rs, 2, 600, lo=4, hi=900)
    want, _ = oracle.pyramid_roi_align(fmaps, props, 1024, 1024, pool[0], pool[1])
    pr = cu(props)
    order = roi_processing_order(pr, [1024, 1024, 3])
    _pyramid(fmaps, props, pool, order=order)
    bad = host(order).copy()
    skipped = [int(bad[3]), int(bad[700]), int(bad[10])]
    bad[3], bad[700] = -1, 5000
    bad[10] = bad[11]
    keep = np.ones(1200, bool)
    keep[skipped] = False
    for md, od in COMBOS:
        out = torch.full((1, 1200, pool[0], pool[1], 256), -7.0, dtype=od, device="cuda")
        got = got_f32(pyramid_roi_align(maps_as(fmaps, md), pr, [1024, 1024], pool, out=out, order=cu(bad.astype(np.int32))), od)
        assert_bits(got[0, keep], rounded(want, od)[0, keep], f"{md} -> {od}: rows of the visited ROIs")
        assert (got[0, ~keep] == -7.0).all(), "rows of skipped ROIs must stay untouched"


@gpu
@pytest.mark.parametrize("combo", COMBOS, ids=IDS)
def test_bf16_without_workspace_static_round_robin(_cuda, combo):
    """od_pyramid_roi_align_forward (no workspace): static round robin in index order, same bits."""
    from objectdetection_b200 import _lib
    md, od = combo
    rs = np.random.RandomState(31)
    fmaps = [bf16_values(rs.random_sample((2, s, s, 256))) for s in (64, 32, 16, 8)]
    props = _synth.rois_log_uniform(rs, 2, 400, lo=4, hi=900)
    want, wlv = oracle.pyramid_roi_align(fmaps, props, 1024, 1024, 14, 14)
    L, dl = _lib.lib(), _lib.DL()
    fm, rois = maps_as(fmaps, md), cu(props)
    out = torch.empty((1, 800, 14, 14, 256), dtype=od, device="cuda")
    lv = torch.empty((2, 400), dtype=torch.int32, device="cuda")
    ptrs = (ctypes.c_void_p * 4)(*[dl(f) for f in fm])
    _lib.check(L.od_pyramid_roi_align_forward(ptrs, 4, 2, dl(rois), 1024, 1024, 14, 14, dl(out), dl(lv),
                                              _lib.stream_ptr(rois.device)), "od_pyramid_roi_align_forward")
    assert_bits(got_f32(out, od), rounded(want, od), "pooled (static round robin)")
    assert np.array_equal(host(lv), wlv)
    assert _counters_zeroed()


@gpu
@pytest.mark.parametrize("D", [256, 8])
def test_bf16_crop_and_resize_box_ind_and_extrapolation(_cuda, D):
    """Out-of-range box_ind leaves the rows untouched; the extrapolation value is rounded like every output value
    (1/3 is not a bf16 value). D = 256 runs crop_rows_kernel for the larger crops, D = 8 crop_bins_kernel<512, ...>."""
    from objectdetection_b200.maskrcnn import crop_and_resize
    rs = np.random.RandomState(12)
    img = bf16_values(rs.random_sample((3, 19, 23, D)))
    boxes = np.concatenate([np.array([[0, 0, 1, 1], [0.1, 0.2, 0.7, 0.9], [0.3, 0.3, 0.3, 0.3], [-0.2, -0.1, 0.5, 0.5],
                                      [0.5, 0.5, 1.3, 1.2], [0.9, 0.8, 0.1, 0.2], [0, 0, 0, 0], [0.25, 0.5, 0.75, 1.0]], f32),
                            _synth.random_boxes(rs, 24, flip=True)])
    bi = rs.randint(0, 3, boxes.shape[0]).astype(np.int32)
    bi[7], bi[9] = 5, -1
    for extrap in (0.5, 1.0 / 3.0):
        for crop in ((7, 7), (14, 14), (1, 3), (16, 9)):
            out0 = np.full((boxes.shape[0], crop[0], crop[1], D), -7.0, f32)
            want = oracle.crop_and_resize(img, boxes, bi, crop[0], crop[1], extrapolation=extrap, out=out0.copy())
            for md, od in COMBOS:
                got = got_f32(crop_and_resize(cu(img).to(md), cu(boxes), cu(bi), crop, extrapolation_value=extrap,
                                              out=cu(out0).to(od)), od)
                assert_bits(got, rounded(want, od), f"{md} -> {od} crop {crop} extrapolation {extrap}")
                assert (got[7] == -7.0).all() and (got[9] == -7.0).all()


@gpu
@pytest.mark.parametrize("D", [8, 24, 40])
def test_bf16_thin_and_non_power_of_two_depth(_cuda, D):
    """D / 8 = 1, 3, 5 bf16 units per pixel: crop_bins_kernel<512, ...> with and without the power-of-two split."""
    rs = np.random.RandomState(900 + D)
    fmaps = [bf16_values(rs.random_sample((2, s, s, D))) for s in (64, 32, 16, 8)]
    props = _synth.rois_with_edge_cases(rs, 2, 120)
    for pool in ([7, 7], [14, 14], [3, 5]):
        _pyramid(fmaps, props, pool)


# ------------------------------------------------------------------ non-finite and range edges
def _edge_image(rs, D):
    """Feature values that exercise the conversions: inf / NaN, values above the largest bf16 (fp32 maps only: they
    round to inf) and below the smallest normal bf16 (they round to bf16 subnormals or zero)."""
    img = rs.random_sample((2, 11, 13, D)).astype(f32)
    img[0, 2, 3, :] = np.inf
    img[0, 4, 5, ::3] = -np.inf
    img[1, 6, 7, 1::2] = np.nan
    img[1, 0:4, :, :] = f32(3.4e38) * rs.choice([-1, 1], size=(4, 13, D)).astype(f32)    # rounds past the bf16 max
    img[0, 6:, :, :] = (rs.random_sample((5, 13, D)) * 2e-38).astype(f32)                 # < smallest normal (1.18e-38)
    img[0, 8:, :, ::4] = f32(1e-40)                                                       # fp32 subnormal
    return img


@gpu
@pytest.mark.parametrize("D", [256, 8])
def test_bf16_non_finite_and_range_edges(_cuda, D):
    from objectdetection_b200.maskrcnn import crop_and_resize
    rs = np.random.RandomState(2024 + D)
    img = _edge_image(rs, D)
    boxes = np.concatenate([np.array([[0, 0, 1, 1], [0.1, 0.2, 0.9, 0.7], [0.0, 0.0, 0.4, 0.4], [0.6, 0.6, 1.0, 1.0]], f32),
                            _synth.random_boxes(rs, 20)])
    bi = np.array([0, 1] * (boxes.shape[0] // 2), np.int32)
    for md, od in COMBOS:
        maps = rounded(img, md)                            # what the kernel reads, as fp32
        for crop in ((14, 14), (7, 7)):
            want = oracle.crop_and_resize(maps, boxes, bi, crop[0], crop[1])
            ref = host(crop_and_resize(cu(maps), cu(boxes), cu(bi), crop))
            assert_bits(ref, want, f"fp32 path {crop}")
            got = got_f32(crop_and_resize(cu(img).to(md), cu(boxes), cu(bi), crop, out_dtype=od), od)
            assert_bits(got, rounded(want, od), f"{md} -> {od} crop {crop}")
            if od == BF16 and md == F32:
                # from halfway between the largest bf16 (0x7F7F) and the next power of two up, RNE gives inf
                big = np.isfinite(want) & (np.abs(want) >= np.array(0x7F7F8000, np.uint32).view(f32))
                assert big.any() and np.isinf(got[big]).all(), "fp32 results above the largest bf16 round to inf"
            small = (np.abs(want) < 1.1754944e-38) & (want != 0)
            assert small.any()
            if od == BF16:
                assert (got[small] != 0).any(), "results below the smallest normal bf16 keep bf16 subnormals"


# ------------------------------------------------------------------ dispatch
def _dispatch_worker():
    """Traces the 14x14 and 7x7 pooling of every new dtype pair and prints the kernel names as JSON."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    from objectdetection_b200.maskrcnn import pyramid_roi_align
    rs = np.random.RandomState(3)
    fm = [cu(rs.random_sample((2, s, s, 256)).astype(f32)) for s in (64, 32, 16, 8)]
    pr = cu(_synth.rois_log_uniform(rs, 2, 300, lo=4, hi=900))
    res = {}
    for (md, od), cid in zip(COMBOS, IDS):
        maps = [f.to(md) for f in fm]
        for P in (14, 7):
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA], acc_events=True) as prof:
                pyramid_roi_align(maps, pr, [1024, 1024], [P, P], out_dtype=od)
                torch.cuda.synchronize()
            res[f"{cid}/{P}"] = [e.name for e in prof.events() if e.device_type == DeviceType.CUDA
                                 and not e.name.startswith(("Memcpy", "Memset"))]
    json.dump(res, sys.stdout)


@gpu
def test_bf16_dispatch_selects_the_bf16_overloads(_cuda):
    """D = 256 at 14x14 runs the bf16 overload of crop_rows_kernel, 7x7 that of crop_bins_kernel; no fp32 sibling runs.
    Traced in a process of its own: in a process that has run many other GPU tests, a profiler session has come back
    without any device activity."""
    flags = ["-s"] if sys.flags.no_user_site else []
    r = subprocess.run([sys.executable, *flags, os.path.abspath(__file__), "--dispatch"], cwd=ROOT, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    res = json.loads(r.stdout)
    for cid in IDS:
        names = res[f"{cid}/14"]
        assert names, f"{cid}: the CUDA kernel trace is empty"
        assert_launched(names, must=["crop_rows_kernel<"], must_not=["od::crop_rows_kernel(", "crop_bins_kernel"])
        assert all("__nv_bfloat16" in n for n in names if "crop_rows_kernel" in n), names
        names = res[f"{cid}/7"]
        assert names, f"{cid}: the CUDA kernel trace is empty"
        assert_launched(names, must=["crop_bins_kernel<"], must_not=["od::crop_bins_kernel<32,", "crop_rows_kernel"])
        assert all("__nv_bfloat16" in n for n in names if "crop_bins_kernel" in n), names


# ------------------------------------------------------------------ Python interface
@gpu
def test_bf16_maps_default_arguments_equal_the_fp32_upcast(_cuda):
    """bf16 maps with default arguments: fp32 pooled rows, bit for bit those of ``[f.float() for f in maps]`` (what the
    call used to compute by upcasting), without the fp32 copy of the pyramid."""
    from objectdetection_b200 import MaskRCNN
    from objectdetection_b200.maskrcnn import pyramid_roi_align
    rs = np.random.RandomState(11)
    maps = [torch.rand((2, s, s, 256), device="cuda").to(BF16) for s in (256, 128, 64, 32)]
    props = cu(_synth.rois_log_uniform(rs, 2, 1000))
    for pool in ([7, 7], [14, 14]):
        want = pyramid_roi_align([f.float() for f in maps], props, [1024, 1024], pool)
        m = MaskRCNN(image_shape=[1024, 1024, 3], pool_shape=pool, num_classes=4, levels=[2, 3, 4, 5], proposals=props,
                     feature_maps=maps)
        got = m.get_pooled_rois()
        assert got.dtype == F32
        assert_bits(host(got), host(want), f"MaskRCNN {pool}")
    fp32_pyramid = sum(f.numel() * 4 for f in maps)
    out = torch.empty((1, 2000, 14, 14, 256), dtype=F32, device="cuda")
    pyramid_roi_align(maps, props, [1024, 1024], [14, 14], out=out)        # workspace allocated once, outside the window
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    pyramid_roi_align(maps, props, [1024, 1024], [14, 14], out=out)
    torch.cuda.synchronize()
    extra = torch.cuda.max_memory_allocated() - base
    assert extra < fp32_pyramid // 4, f"the call allocated {extra} bytes (an fp32 copy of the pyramid is {fp32_pyramid})"


@gpu
def test_bf16_maps_the_bf16_kernels_do_not_take_are_converted_as_before(_cuda):
    """bf16 maps with D % 8 != 0 (D = 4, 12) or at an 8-byte offset: with default arguments the call converts them to
    fp32, as it always did, and returns what pooling ``[f.float() for f in maps]`` returns."""
    from objectdetection_b200.maskrcnn import crop_and_resize, pyramid_roi_align
    rs = np.random.RandomState(17)
    pr = cu(_synth.rois_log_uniform(rs, 2, 200))
    for D in (4, 12):
        maps = [cu(rs.random_sample((2, s, s, D)).astype(f32)).to(BF16) for s in (64, 32, 16, 8)]
        for pool in ([7, 7], [14, 14]):
            want = host(pyramid_roi_align([f.float() for f in maps], pr, [1024, 1024], pool))
            assert_bits(host(pyramid_roi_align(maps, pr, [1024, 1024], pool)), want, f"D = {D} {pool}")
        img = maps[1]
        boxes, bi = cu(_synth.random_boxes(rs, 6)), cu(np.array([0, 1, 0, 1, 0, 1], np.int32))
        assert_bits(host(crop_and_resize(img, boxes, bi, (7, 7))), host(crop_and_resize(img.float(), boxes, bi, (7, 7))),
                    f"crop_and_resize D = {D}")
    # contiguous bf16 views 8 bytes past a 16-byte boundary
    flat = [torch.rand(2 * s * s * 256 + 4, device="cuda").to(BF16) for s in (64, 32, 16, 8)]
    maps = [f[4:].view(2, s, s, 256) for f, s in zip(flat, (64, 32, 16, 8))]
    assert all(m.data_ptr() % 16 == 8 for m in maps)
    want = host(pyramid_roi_align([f.float() for f in maps], pr, [1024, 1024], [7, 7]))
    assert_bits(host(pyramid_roi_align(maps, pr, [1024, 1024], [7, 7])), want, "maps at an 8-byte offset")


@gpu
def test_bf16_output_dtype_selection(_cuda):
    from objectdetection_b200 import MaskRCNN
    from objectdetection_b200.maskrcnn import crop_and_resize, pyramid_roi_align

    class _Bf16Pooled(MaskRCNN):
        pooled_dtype = BF16

    rs = np.random.RandomState(13)
    fm = [cu(bf16_values(rs.random_sample((1, s, s, 256)))) for s in (64, 32, 16, 8)]
    pr = cu(_synth.rois_log_uniform(rs, 1, 50))
    ref = pyramid_roi_align(fm, pr, [1024, 1024], [7, 7])
    assert ref.dtype == F32
    for maps in (fm, [f.to(BF16) for f in fm]):
        assert pyramid_roi_align(maps, pr, [1024, 1024], [7, 7]).dtype == F32
        assert pyramid_roi_align(maps, pr, [1024, 1024], [7, 7], out_dtype=BF16).dtype == BF16
        out = torch.empty((1, 50, 7, 7, 256), dtype=BF16, device="cuda")
        assert pyramid_roi_align(maps, pr, [1024, 1024], [7, 7], out=out, out_dtype=F32) is out   # out wins
        m = _Bf16Pooled([1024, 1024, 3], [7, 7], 4, [2, 3, 4, 5], pr, maps)
        assert m.get_pooled_rois().dtype == BF16
        assert_bits(host(m.get_pooled_rois().float()), bf16_values(host(ref)), "pooled_dtype=bfloat16")
    boxes, bi = cu(np.array([[0.1, 0.1, 0.8, 0.9]], f32)), cu(np.zeros(1, np.int32))
    img = fm[1]
    assert crop_and_resize(img, boxes, bi, (7, 7)).dtype == F32
    assert crop_and_resize(img.to(BF16), boxes, bi, (7, 7)).dtype == F32
    assert crop_and_resize(img.to(BF16), boxes, bi, (7, 7), out_dtype=BF16).dtype == BF16
    # a list of maps that do not share one dtype is converted to fp32, as before
    mixed = [fm[0].to(BF16)] + fm[1:]
    assert_bits(host(pyramid_roi_align(mixed, pr, [1024, 1024], [7, 7])),
                host(pyramid_roi_align([f.float() for f in mixed], pr, [1024, 1024], [7, 7])), "mixed map dtypes")


# ------------------------------------------------------------------ refusals (no GPU)
BF, F16, FL = (4, 16), (2, 16), (2, 32)


def _refusal_cases():
    """(case id, entry, {tensor: (dtype, shape, byte_offset)} overrides, expected status, argument the detail names)."""
    C = []
    pyr = ["od_pyramid_roi_align_forward", "od_pyramid_roi_align_forward_ws", "od_pyramid_roi_align_forward_ordered"]
    for e in pyr + ["od_crop_and_resize"]:
        m0, m1, o = ("image", None, "out") if e == "od_crop_and_resize" else ("fmaps[0]", "fmaps[1]", "pooled")
        maps = [m0] + ([m1] if m1 else [])
        both = lambda dt: {m: (dt,) for m in maps}  # noqa: E731
        for md, od in ((BF, FL), (FL, BF), (BF, BF)):
            C.append((f"{e}-{md}-{od}-accepted", e, {**both(md), o: (od,)}, ACCEPTED, None))
        C.append((f"{e}-f16-maps", e, both(F16), -2, m0))
        C.append((f"{e}-f16-out", e, {o: (F16,)}, -2, o))
        C.append((f"{e}-bf16-maps-f16-out", e, {**both(BF), o: (F16,)}, -2, o))
        C.append((f"{e}-bf16-maps-depth12", e, {**{m: (BF, 12) for m in maps}, o: (FL, 12)}, -3, None))
        C.append((f"{e}-bf16-out-depth12", e, {**{m: (FL, 12) for m in maps}, o: (BF, 12)}, -3, None))
        C.append((f"{e}-bf16-maps-offset8", e, {**both(BF), m0: (BF, None, 8)}, -5, m0))
        C.append((f"{e}-bf16-out-offset8", e, {o: (BF, None, 8)}, -5, o))
        if m1:
            C.append((f"{e}-mixed-levels", e, {m0: (BF,), m1: (FL,)}, -2, "fmaps[l]"))
            C.append((f"{e}-mixed-levels-f32-first", e, {m0: (FL,), m1: (BF,)}, -2, "fmaps[l]"))
    C.append(("od_roi_pool_forward-bf16-map", "od_roi_pool_forward", {"feature_map": (BF,)}, -2, "feature_map"))
    C.append(("od_roi_pool_forward-bf16-out", "od_roi_pool_forward", {"out": (BF,)}, -2, "out"))
    return C


REFUSALS = _refusal_cases()


def _worker():
    if os.environ.get("CUDA_VISIBLE_DEVICES") != "":
        raise SystemExit("refusing to run: CUDA_VISIBLE_DEVICES must be empty")
    from objectdetection_b200 import _lib
    if torch.cuda.device_count() != 0:
        raise SystemExit("refusing to run: a CUDA device is visible")
    L = _lib.lib()
    base = {"fmaps[0]": (2, 4, 4, 8), "fmaps[1]": (2, 2, 2, 8), "rois": (2, 3, 4), "pooled": (6, 2, 2, 8),
            "image": (2, 4, 4, 8), "boxes": (3, 4), "box_ind": (3,), "out": (3, 2, 2, 8),
            "feature_map": (2, 4, 4, 8), "proposals": (3, 5), "roi_level": (2, 3)}
    rp_out = (3, 7, 7, 8)
    keep = []

    def tensor(name, over, ptr, entry):
        dt, shape, off = (over + (None, None, None))[:3] if over else (None, None, None)
        sh = list(rp_out if (entry == "od_roi_pool_forward" and name == "out") else base[name])
        if shape is not None:
            sh[-1] = shape
        t = DLTensor()
        t.data = ptr
        t.device.device_type, t.device.device_id = kDLCUDA, 0
        t.ndim = len(sh)
        t.dtype.code, t.dtype.bits = dt or ((0, 32) if name in ("box_ind", "roi_level") else FL)
        t.dtype.lanes = 1
        a = (ctypes.c_int64 * len(sh))(*sh)
        t.shape = a
        t.byte_offset = off or 0
        keep.extend([a, t])
        return ctypes.cast(ctypes.pointer(t), ctypes.c_void_p).value

    out = {}
    for cid, entry, over, _, _ in REFUSALS:
        names = {"od_crop_and_resize": ["image", "boxes", "box_ind", "out"],
                 "od_roi_pool_forward": ["feature_map", "proposals", "out"]}.get(entry, ["fmaps[0]", "fmaps[1]", "rois",
                                                                                          "pooled", "roi_level"])
        t = {n: tensor(n, over.get(n), 0x10000000 * (i + 1), entry) for i, n in enumerate(names)}
        before = L.od_launch_count()
        if entry == "od_crop_and_resize":
            st = L.od_crop_and_resize(t["image"], t["boxes"], t["box_ind"], 2, 2, 0.0, t["out"], None)
        elif entry == "od_roi_pool_forward":
            st = L.od_roi_pool_forward(t["feature_map"], t["proposals"], 64.0, 64.0, t["out"], None)
        else:
            fm = (ctypes.c_void_p * 2)(t["fmaps[0]"], t["fmaps[1]"])
            args = (fm, 2, 2, t["rois"], 64, 64, 2, 2, t["pooled"], t["roi_level"])
            if entry == "od_pyramid_roi_align_forward":
                st = L.od_pyramid_roi_align_forward(*args, None)
            elif entry == "od_pyramid_roi_align_forward_ws":
                st = L.od_pyramid_roi_align_forward_ws(*args, 0x7F0000000000, 1 << 40, None)
            else:
                st = L.od_pyramid_roi_align_forward_ordered(*args, None, 0x7F0000000000, 1 << 40, None)
        out[cid] = [st, L.od_last_error_detail().decode(errors="replace"), L.od_launch_count() != before]
    json.dump(out, sys.stdout)


@pytest.fixture(scope="module")
def refusals():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    flags = ["-s"] if sys.flags.no_user_site else []
    r = subprocess.run([sys.executable, *flags, os.path.abspath(__file__), "--worker"], env=env, cwd=ROOT,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    return json.loads(r.stdout)


@pytest.mark.parametrize("case", REFUSALS, ids=[c[0] for c in REFUSALS])
def test_bf16_validation(refusals, case):
    cid, _, _, expected, names = case
    status, detail, launched = refusals[cid]
    assert status == expected, f"{cid}: status {status}, expected {expected} ({detail})"
    if expected != ACCEPTED:
        assert not launched, f"{cid}: refused with {status} after a launch"
    if names:
        names = "fmaps[l]" if names.startswith("fmaps") else names     # the levels are reported as fmaps[l]
        assert names in detail, f"{cid}: detail {detail!r} does not name {names}"


if __name__ == "__main__" and sys.argv[1:] == ["--worker"]:
    _worker()
if __name__ == "__main__" and sys.argv[1:] == ["--dispatch"]:
    _dispatch_worker()
