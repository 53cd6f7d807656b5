"""Kernel dispatch: each C entry point picks one of several kernels (or template instantiations) from the input's shape.
The tests here reach the branches that the benchmark-sized inputs of test_gpu_parity.py never take, check the outputs
against the CPU oracle as strictly as test_gpu_parity.py does, and read from a CUDA kernel trace that the intended
kernel ran and its sibling did not, so that a retuned threshold cannot silently turn a test into a test of another
branch. Non-power-of-two depths are also compared with the float64 crop_and_resize of tests/_f64_refs.py.

KERNEL_PATHS names, for every __global__ kernel in objectdetection_b200/csrc, the test that launches it;
test_kernel_paths_cover_every_kernel (no GPU) fails when a kernel is missing from it."""
import ctypes
import glob
import os
import re
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import _synth  # noqa: E402
from _f64_refs import crop_and_resize_f64  # noqa: E402

import oracle  # noqa: E402
from objectdetection_b200.config import ShapesConfig, config as Conf  # noqa: E402
from test_gpu_parity import _check_detection, _check_targets, _roi_align_check, assert_bits, cu, host  # noqa: E402

torch = pytest.importorskip("torch")
f32 = np.float32
CSRC = os.path.join(os.path.dirname(HERE), "objectdetection_b200", "csrc")

P, D_ = "test_gpu_parity.py::", "test_gpu_dispatch.py::"
KERNEL_PATHS = {
    # topk.cu
    "topk_collect_kernel": P + "test_topk",
    "topk_hist1_kernel": P + "test_topk",
    "topk_split_kernel": P + "test_topk",
    "topk_tail_kernel": P + "test_topk",
    "topk_tile_sort_kernel": P + "test_topk",
    "topk_merge_emit_kernel": P + "test_topk",
    "sort_u64_smem_kernel": D_ + "test_detection_bitonic_sort_and_gather",
    "bitonic_step_global_kernel": D_ + "test_topk_merge_and_global_sort_boundary",
    "pad_emit_kernel": D_ + "test_topk_merge_and_global_sort_boundary",
    # frcnn.cu
    "frcnn_decode_kernel": P + "test_frcnn_proposals_and_roi_pool",
    "frcnn_rank_gather_kernel": P + "test_frcnn_proposals_and_roi_pool",
    "frcnn_mask_kernel": P + "test_frcnn_proposals_and_roi_pool",
    "frcnn_gather_kernel": P + "test_frcnn_proposals_and_roi_pool",
    "frcnn_emit_kernel": P + "test_frcnn_proposals_and_roi_pool",
    # rpn_targets.cu
    "rpn_anchor_best_kernel<true>": D_ + "test_rpn_targets_fused_per_gt_boundary",
    "rpn_anchor_best_kernel<false>": D_ + "test_rpn_targets_fused_per_gt_boundary",
    "rpn_gt_reduce_kernel": D_ + "test_rpn_targets_fused_per_gt_boundary",
    "rpn_gt_best_kernel": D_ + "test_rpn_targets_fused_per_gt_boundary",
    "rpn_label_kernel": P + "test_rpn_targets_golden_and_coco_shape",
    "rpn_label_best_kernel": P + "test_rpn_targets_golden_and_coco_shape",
    "rpn_count_kernel": P + "test_rpn_targets_golden_and_coco_shape",
    "rpn_compact_kernel": P + "test_rpn_targets_golden_and_coco_shape",
    "rpn_perm_kernel": P + "test_rpn_targets_golden_and_coco_shape",
    "rpn_emit_kernel": P + "test_rpn_targets_golden_and_coco_shape",
    # roi_align.cu
    "crop_bins_kernel<32, 2, true, true>": P + "test_roi_pooling_processing_order",
    "crop_bins_kernel<32, 2, true, false>": D_ + "test_roi_align_d256_crop_rows_serves_bounds",
    "crop_bins_kernel<512, 2, true, false>": P + "test_crop_and_resize_generic",
    "crop_bins_kernel<512, 2, false, false>": D_ + "test_roi_align_non_power_of_two_depth",
    "roi_order_kernel": P + "test_roi_pooling_processing_order",
    "crop_rows_kernel": D_ + "test_roi_align_d256_crop_rows_serves_bounds",
    "crop_pool_bins_kernel": D_ + "test_roi_pool_non_power_of_two_depth",
    # nms.cu
    "nms_mask_kernel<true>": D_ + "test_nms_thresholds_zero_one_and_padded_rows",
    "nms_mask_kernel<false>": D_ + "test_nms_negative_threshold",
    "nms_scan_kernel<true>": P + "test_nms",
    # reached in the second round of a two-round NMS; single-round it needs hundreds of images at K > 12600 (GBs of mask)
    "nms_scan_kernel<false>": P + "test_nms_two_rounds_on_clustered_boxes",
    "nms_scan_wide_kernel<true>": D_ + "test_detection_16384_rois_wide_nms_and_finalize_carry",
    "nms_scan_wide_kernel<false>": D_ + "test_nms_wide_scan_without_prefetch",
    "nms_build_keys_kernel": P + "test_nms",
    "nms_gather_sorted_kernel": P + "test_nms",
    "nms_map_back_kernel": P + "test_nms",
    # targets.cu
    "detection_iou_kernel": D_ + "test_detection_targets_large_gt_shared_memory",
    "detection_target_kernel": P + "test_detection_targets_training_config",
    "mask_target_kernel": D_ + "test_mask_targets_both_layouts_non_square",
    # proposal.cu
    "proposal_decode_kernel": P + "test_proposals_coco_shape",
    "rpn_level_scores_kernel": P + "test_proposals_from_rpn_level_outputs",
    "proposal_gather_kernel": P + "test_proposals_coco_shape",
    "apply_box_deltas_kernel": P + "test_apply_box_deltas_and_clip",
    "clip_boxes_kernel": P + "test_apply_box_deltas_and_clip",
    "gen_anchors_norm_kernel": P + "test_gen_anchors_bit_exact",
    "gen_anchors_pixel_kernel": P + "test_gen_anchors_bit_exact",
    "norm_boxes_kernel": "test_gpu_parity_goldens.py::test_norm_boxes_tf_equals_reference_run",
    # losses.cu
    "rpn_loss_class_kernel": P + "test_head_losses",
    "rpn_loss_box_kernel": P + "test_head_losses",
    "rpn_loss_final_kernel": P + "test_head_losses",
    "mrcnn_loss_kernel": P + "test_head_losses",
    # detection.cu
    "det_prepare_kernel": P + "test_detection_coco_shape",
    "det_rank_gather_kernel": D_ + "test_detection_rank_gather_multi_tile",
    "det_gather_kernel": D_ + "test_detection_bitonic_sort_and_gather",
    "det_finalize_kernel": D_ + "test_detection_16384_rois_wide_nms_and_finalize_carry",
    "unmold_kernel": P + "test_unmold_detections_on_device",
}


def _kernels_in_sources():
    names = set()
    for path in glob.glob(os.path.join(CSRC, "*.cu")) + glob.glob(os.path.join(CSRC, "*.cuh")):
        src = open(path).read()
        names |= set(re.findall(r"__global__\s+(?:void\s+)?(?:__launch_bounds__\([^)]*\)\s*)?(?:void\s+)?(\w+)\s*\(", src))
    return names


def test_kernel_paths_cover_every_kernel():
    """Every __global__ kernel has a KERNEL_PATHS entry; every entry names a kernel that exists and a test that exists."""
    kernels = _kernels_in_sources()
    assert len(kernels) > 40, kernels
    covered = {k.split("<")[0] for k in KERNEL_PATHS}
    missing = sorted(kernels - covered)
    assert not missing, f"kernels without a KERNEL_PATHS entry (name the test that launches them): {missing}"
    stale = sorted(covered - kernels)
    assert not stale, f"KERNEL_PATHS entries for kernels that no longer exist: {stale}"
    for kernel, where in KERNEL_PATHS.items():
        fname, test = where.split("::")
        src = open(os.path.join(HERE, fname)).read()
        assert re.search(rf"^def {re.escape(test)}\(", src, re.M), f"{kernel}: {where} does not exist"


# ------------------------------------------------------------------ kernel trace
def _flat(s):
    return re.sub(r"\s+", "", s)


@pytest.fixture
def kernel_trace():
    """trace(fn) -> (fn(), names of the CUDA kernels fn launched, demangled as kineto reports them)."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile

    def trace(fn):
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA], acc_events=True) as prof:
            out = fn()
            torch.cuda.synchronize()
        names = [e.name for e in prof.events() if e.device_type == DeviceType.CUDA
                 and not e.name.startswith(("Memcpy", "Memset"))]
        assert names, "the CUDA kernel trace is empty: torch.profiler recorded no kernel"
        return out, names
    return trace


def assert_launched(names, must=(), must_not=()):
    flat = [_flat(n) for n in names]
    for m in must:
        hit = sorted({n for n, f in zip(names, flat) if _flat(m) in f})
        assert hit, f"{m} was not launched; the trace has {sorted(set(names))}"
        print("launched:", *hit, sep="\n  ")
    for m in must_not:
        hit = sorted({n for n, f in zip(names, flat) if _flat(m) in f})
        assert not hit, f"{m} must not run here, but the trace has {hit}"


@pytest.fixture(scope="module")
def _cuda():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (there is no CPU path)")


# ------------------------------------------------------------------ float64 crop_and_resize
def _assert_close_f64(got, want, ok, what):
    assert ok.mean() > 0.5, f"{what}: only {ok.mean():.3f} of the bins are comparable"
    err = np.abs(got.astype(np.float64) - want)[ok]
    assert err.max() <= 1e-4, f"{what}: max |cuda - fp64| = {err.max():.3e} over {ok.sum()} bins"


def test_crop_and_resize_f64_reference_is_tf():
    """The float64 reference itself, on hand-computed values: corners, centre formula, extrapolation."""
    img = np.arange(12, dtype=np.float64).reshape(1, 3, 4, 1)           # value = 4*y + x
    out, ok = crop_and_resize_f64(img, np.array([[0, 0, 1, 1], [0.5, 0.5, 0.5, 0.5], [-1, 0, 0, 1]]),
                                  np.array([0, 0, 0]), 3, 2, extrapolation=-5.0)
    assert np.array_equal(out[0, :, :, 0], [[0, 3], [4, 7], [8, 11]])
    assert np.allclose(out[1, :, :, 0], 4 * 1 + 1.5)
    assert np.array_equal(out[2, :, :, 0], [[-5, -5], [-5, -5], [0, 3]])
    assert ok[1].all() and not ok[0, 0].any() and not ok[2, 2].any()
    single, _ = crop_and_resize_f64(img, np.array([[0, 0, 1, 1]]), np.array([0]), 1, 1)
    assert single[0, 0, 0, 0] == 4 * 1 + 1.5


# ------------------------------------------------------------------ DetectionLayer
WIN = np.array([[131, 0, 893, 1024], [0, 0, 1024, 1024]], "int32")


def _detection_inputs(seed, N, C=81, boosted=0.9):
    rs = np.random.RandomState(seed)
    props = _synth.rois_log_uniform(rs, 2, N)
    probs, bbox = _synth.head_outputs(rs, 2, N, C, boosted=boosted)
    return props, probs, bbox


def _kept_before_nms(probs, conf):
    return ((probs.argmax(-1) > 0) & (probs.max(-1) > conf.DETECTION_MIN_THRESHOLD)).sum(1)


@pytest.mark.gpu
@pytest.mark.parametrize("N", [4097, 8192])
def test_detection_bitonic_sort_and_gather(_cuda, kernel_trace, N):
    """N > 4096 ROIs: the keys are sorted in shared memory and gathered by det_gather_kernel (num_valid = the last kept
    position) instead of the fused rank sort."""
    props, probs, bbox = _detection_inputs(N, N)
    props[1, N - 300:] = 0
    _, names = kernel_trace(lambda: _check_detection(Conf(), WIN, [1024, 1024, 3], props, probs, bbox))
    assert_launched(names, must=["od::sort_u64_smem_kernel(", "od::det_gather_kernel(", "od::det_finalize_kernel("],
                    must_not=["od::det_rank_gather_kernel(", "od::bitonic_step_global_kernel("])
    assert (_kept_before_nms(probs, Conf()) > 1024).all()


@pytest.mark.gpu
def test_detection_16384_rois_wide_nms_and_finalize_carry(_cuda, kernel_trace):
    """N = 16384 (the cap), B = 2: class-grouped NMS over K = N boxes through the cooperative wide scan, and more than
    1024 kept ROIs per image, so det_finalize_kernel's prefix count carries tile_base across 1024-element tiles (its
    dynamic shared memory is 192 KiB)."""
    N = 16384
    props, probs, bbox = _detection_inputs(7, N)
    conf = Conf()
    det, names = kernel_trace(lambda: _check_detection(conf, WIN, [1024, 1024, 3], props, probs, bbox))
    assert_launched(names, must=["od::sort_u64_smem_kernel(", "od::det_gather_kernel(", "od::nms_scan_wide_kernel<true>(",
                                 "od::det_finalize_kernel("],
                    must_not=["od::det_rank_gather_kernel(", "od::nms_scan_kernel<"])
    assert (_kept_before_nms(probs, conf) > 1024).all()
    assert ((det[:, :, 4] > 0).sum(1) == conf.DETECTION_POST_NMS_INSTANCES).all()


@pytest.mark.gpu
@pytest.mark.parametrize("N", [2000, 4096])
def test_detection_rank_gather_multi_tile(_cuda, kernel_trace, N):
    """1024 < N <= 4096: det_rank_gather_kernel counts each key's rank over several 1024-key tiles."""
    props, probs, bbox = _detection_inputs(N + 1, N, boosted=0.75)
    props[1, N - 100:] = 0
    _, names = kernel_trace(lambda: _check_detection(Conf(), WIN, [1024, 1024, 3], props, probs, bbox))
    assert_launched(names, must=["od::det_rank_gather_kernel("],
                    must_not=["od::det_gather_kernel(", "od::sort_u64_smem_kernel("])
    assert (_kept_before_nms(probs, Conf()) > 1024).all()


@pytest.mark.gpu
@pytest.mark.parametrize("C", [1, 2])
def test_detection_one_and_two_classes(_cuda, kernel_trace, C):
    """C = 1: only the background class, nothing can be kept. C = 2: every kept ROI is in the one NMS group."""
    rs = np.random.RandomState(40 + C)
    N = 1000
    props = _synth.rois_log_uniform(rs, 2, N)
    if C == 1:
        probs = np.ones((2, N, 1), f32)
        bbox = rs.normal(0, 1, (2, N, 1, 4)).astype(f32)
    else:
        probs, bbox = _synth.head_outputs(rs, 2, N, C, boosted=0.6)
    det, names = kernel_trace(lambda: _check_detection(Conf(), WIN, [1024, 1024, 3], props, probs, bbox))
    assert_launched(names, must=["od::det_prepare_kernel(", "od::det_rank_gather_kernel(", "od::det_finalize_kernel("])
    if C == 1:
        assert not det.any()
    else:
        n = (det[:, :, 4] > 0).sum(1)
        assert (n > 0).all() and set(np.unique(det[:, :, 4])) <= {0.0, 1.0}


# ------------------------------------------------------------------ NMS
def _clustered_boxes(rs, K, n_clusters=300):
    centers, sizes = rs.uniform(0.1, 0.9, (n_clusters, 2)), rs.uniform(0.02, 0.1, (n_clusters, 2))
    which = rs.randint(0, n_clusters, K)
    c = centers[which] + rs.normal(0, 0.004, (K, 2))
    hw = sizes[which] * np.exp(rs.normal(0, 0.06, (K, 2)))
    return np.concatenate([c - hw / 2, c + hw / 2], -1).astype(f32)


def _check_nms(boxes, scores, max_out, thr, nv):
    from objectdetection_b200.proposals import non_max_suppression
    keep, num = non_max_suppression(cu(boxes), cu(scores), max_out, thr, num_valid=nv)
    keep, num = host(keep), host(num)
    wants = []
    for b in range(boxes.shape[0]):
        want = oracle.nms(boxes[b, :nv[b]], scores[b, :nv[b]], max_out, thr)
        assert num[b] == want.shape[0], (b, num[b], want.shape[0])
        assert np.array_equal(keep[b, :num[b]], want) and np.all(keep[b, num[b]:] == -1)
        wants.append(want)
    return wants


@pytest.mark.gpu
def test_nms_wide_scan_without_prefetch(_cuda, kernel_trace):
    """B = 8 images of K = 20000 boxes, max_out = K: the per-image slice of the cooperative scan is too wide for the
    diagonal block in shared memory (18 words on 148 SMs), so nms_scan_wide_kernel<false> runs. Clustered and sparse
    images, ragged num_valid."""
    B, K = 8, 20000
    rs = np.random.RandomState(8)
    boxes = np.stack([_clustered_boxes(rs, K) if b % 2 == 0 else
                      _synth.rois_log_uniform(rs, 1, K, image=4096, lo=4, hi=48)[0] for b in range(B)])
    scores = rs.random_sample((B, K)).astype(f32)
    nv = np.array([K, K - 1777, 64, K, 12345, K, 1, K], np.int32)
    wants, names = kernel_trace(lambda: _check_nms(boxes, scores, K, 0.5, nv))
    assert_launched(names, must=["od::nms_scan_wide_kernel<false>(", "od::nms_mask_kernel<true>("],
                    must_not=["od::nms_scan_wide_kernel<true>(", "od::nms_scan_kernel<"])
    assert wants[0].shape[0] < 2000 and wants[1].shape[0] > 10000      # both regimes: few and many survivors


@pytest.mark.gpu
def test_nms_negative_threshold(_cuda, kernel_trace):
    """iou_threshold < 0: the exact kernel (no candidate pre-pass); every IoU, zero included, exceeds it."""
    rs = np.random.RandomState(11)
    K = 300
    boxes = np.stack([_synth.random_boxes(rs, K, flip=True) for _ in range(2)])
    boxes[0, 3] = 0                                                    # zero area
    boxes[1, 7, 2:] = boxes[1, 7, :2]
    scores = (rs.randint(0, 50, (2, K)) / 50).astype(f32)
    wants, names = kernel_trace(lambda: _check_nms(boxes, scores, K, -0.1, np.array([K, 250], np.int32)))
    assert_launched(names, must=["od::nms_mask_kernel<false>("], must_not=["od::nms_mask_kernel<true>("])
    assert [w.shape[0] for w in wants] == [1, 1]


@pytest.mark.gpu
@pytest.mark.parametrize("thr", [0.0, 1.0])
def test_nms_thresholds_zero_one_and_padded_rows(_cuda, kernel_trace, thr):
    """Thresholds 0 (any overlap suppresses) and 1 (nothing suppresses, identical boxes included: IoU 1 is not > 1) on
    the candidate kernel, with max_output_size = 1000 > K = 300: rows beyond the kept ones are -1."""
    rs = np.random.RandomState(12)
    K = 300
    boxes = np.stack([_synth.random_boxes(rs, K, flip=True) for _ in range(2)])
    boxes[0, 5] = boxes[0, 6]
    boxes[0, 10, 2:] = boxes[0, 10, :2]
    boxes[1, 20] = boxes[1, 21] = boxes[1, 22]
    scores = (rs.randint(0, 100, (2, K)) / 100).astype(f32)
    wants, names = kernel_trace(lambda: _check_nms(boxes, scores, 1000, thr, np.array([K, 299], np.int32)))
    assert_launched(names, must=["od::nms_mask_kernel<true>("], must_not=["od::nms_mask_kernel<false>("])
    if thr == 1.0:
        assert [w.shape[0] for w in wants] == [K, 299]
    else:
        assert all(0 < w.shape[0] < 100 for w in wants)


# ------------------------------------------------------------------ ROIAlign / crop_and_resize / roi_pool
def _pyramid_f64(fmaps, props, pool):
    """PyramidROIAlign in float64: oracle.roi_level picks the level, crop_and_resize_f64 samples it."""
    B, N = props.shape[:2]
    lv = oracle.roi_level(props, 1024, 1024)
    out = np.zeros((B * N,) + tuple(pool) + (fmaps[0].shape[-1],))
    ok = np.zeros((B * N,) + tuple(pool), bool)
    for b in range(B):
        for level in range(2, 6):
            sel = np.nonzero(lv[b] == level)[0]
            if sel.size:
                o, k = crop_and_resize_f64(fmaps[level - 2][b:b + 1], props[b, sel], np.zeros(sel.size, np.int32), *pool)
                out[b * N + sel], ok[b * N + sel] = o, k
    return out, ok


@pytest.mark.gpu
@pytest.mark.parametrize("D", [12, 20, 260])
def test_roi_align_non_power_of_two_depth(_cuda, kernel_trace, D):
    """D / 4 not a power of two: crop_bins_kernel<512, 2, false, false> splits elements into (bin, channel) by division.
    PyramidROIAlign (7x7, 14x14) and crop_and_resize (with skipped crops) bit-exact against the oracle and within 1e-4
    of a float64 crop_and_resize."""
    from objectdetection_b200.maskrcnn import crop_and_resize
    rs = np.random.RandomState(D)
    fmaps = [rs.random_sample((2, s, s, D)).astype(f32) for s in (64, 32, 16, 8)]
    props = _synth.rois_with_edge_cases(rs, 2, 200)
    kernel = "od::crop_bins_kernel<512, 2, false, false>("
    for pool in ([7, 7], [14, 14]):
        got, names = kernel_trace(lambda: _roi_align_check(fmaps, props, 1024, pool))
        assert_launched(names, must=[kernel], must_not=["od::crop_rows_kernel(", "od::crop_bins_kernel<32,"])
        want, ok = _pyramid_f64(fmaps, props, pool)
        _assert_close_f64(got[0], want, ok, f"pyramid D={D} {pool}")
    img = rs.random_sample((3, 19, 23, D)).astype(f32)
    boxes = np.concatenate([props[0, :13], _synth.random_boxes(rs, 40, flip=True)])
    bi = rs.randint(0, 3, boxes.shape[0]).astype(np.int32)
    bi[20], bi[30] = 3, -1                                                   # out of range: crop left untouched
    for crop in ((7, 7), (14, 14), (1, 1), (1, 3), (16, 9)):
        out0 = np.full((boxes.shape[0], crop[0], crop[1], D), -7.0, f32)
        got, names = kernel_trace(lambda: host(crop_and_resize(cu(img), cu(boxes), cu(bi), crop, extrapolation_value=0.5,
                                                               out=cu(out0))))
        assert_launched(names, must=[kernel])
        assert_bits(got, oracle.crop_and_resize(img, boxes, bi, crop[0], crop[1], extrapolation=0.5, out=out0.copy()),
                    f"crop {crop} D={D}")
        assert (got[20] == -7.0).all() and (got[30] == -7.0).all()
        want, ok = crop_and_resize_f64(img, boxes, bi, *crop, extrapolation=0.5)
        _assert_close_f64(got, want, ok, f"crop {crop} D={D}")


@pytest.mark.gpu
def test_roi_pool_non_power_of_two_depth(_cuda, kernel_trace):
    """Faster R-CNN roi_pool (14x14 crop, 2x2 max) at D = 20: bit-exact against the oracle, within 1e-4 of float64."""
    from objectdetection_b200 import fasterrcnn
    rs = np.random.RandomState(20)
    D, h, w = 20, 38, 63
    fmap = rs.random_sample((1, h, w, D)).astype(f32)
    xy1 = rs.uniform(-20, 900, (150, 2))
    wh = rs.uniform(0, 300, (150, 2))
    rois = np.concatenate([np.zeros((150, 1)), xy1, xy1 + wh], 1).astype(f32)       # (batch, x1, y1, x2, y2) pixels
    rois[0, 1:] = [0, 0, 1000, 600]
    rois[1, 1:] = [500, 300, 500, 300]
    rois[2, 1:] = [700, 100, 200, 500]                                              # flipped
    got, names = kernel_trace(lambda: host(fasterrcnn.roi_pool(cu(fmap), cu(rois), (600, 1000, 3))))
    assert_launched(names, must=["od::crop_pool_bins_kernel("])
    assert_bits(got, oracle.roi_pool(fmap, rois, 600.0, 1000.0), "roi_pool D=20")
    boxes = np.stack([rois[:, 2] / 600.0, rois[:, 1] / 1000.0, rois[:, 4] / 600.0, rois[:, 3] / 1000.0], 1)
    crops, ok = crop_and_resize_f64(fmap, boxes, np.zeros(150, np.int32), 14, 14)
    want = crops.reshape(150, 7, 2, 7, 2, D).max(axis=(2, 4))
    _assert_close_f64(got, want, ok.reshape(150, 7, 2, 7, 2).all(axis=(2, 4)), "roi_pool D=20")


@pytest.mark.gpu
@pytest.mark.parametrize("pool,rows", [([1, 14], True), ([14, 1], True), ([16, 14], True), ([10, 10], True),
                                       ([9, 9], False), ([17, 14], False)])
def test_roi_align_d256_crop_rows_serves_bounds(_cuda, kernel_trace, pool, rows):
    """The bounds of crop_rows_serves at D = 256: pool height <= 16, width <= 14 and max(height, width) >= 10 take the
    TMA-staged row kernel; just outside them the flat per-bin kernel runs. Same edge-case ROIs, bit-exact either way."""
    rs = np.random.RandomState(4321 + 100 * pool[0] + pool[1])
    fmaps = [rs.random_sample((2, s, s, 256)).astype(f32) for s in (64, 32, 16, 8)]
    props = _synth.rois_with_edge_cases(rs, 2, 160)
    _, names = kernel_trace(lambda: _roi_align_check(fmaps, props, 1024, pool))
    if rows:
        assert_launched(names, must=["od::crop_rows_kernel("], must_not=["od::crop_bins_kernel<"])
    else:
        assert_launched(names, must=["od::crop_bins_kernel<32, 2, true, false>("], must_not=["od::crop_rows_kernel("])


# ------------------------------------------------------------------ DetectionTargetLayer
def _many_gt_inputs(rs, B, N, G, n_pad=200):
    """target inputs with G GT boxes per image, most of them valid: random boxes, one in ten a jittered copy of a
    proposal (spread over all GT rows, so that assigned GT indices reach far into the shared-memory table), one in
    twenty with class 0 (compacted away), and the last 50 rows padding."""
    props = _synth.rois_log_uniform(rs, B, N)
    props[:, N - n_pad:] = 0
    gt = _synth.rois_log_uniform(rs, B, G)
    cls = rs.randint(1, 81, (B, G)).astype(np.int32)
    for b in range(B):
        copies = rs.choice(G, G // 10, replace=False)
        gt[b, copies] = props[b, rs.randint(0, N - n_pad, copies.size)] + rs.normal(0, 0.01, (copies.size, 4)).astype(f32)
        cls[b, rs.random_sample(G) < 0.05] = 0
    cls[:, G - 50:] = 0
    gt[:, G - 50:] = 0
    pp = np.stack([rs.permutation(N) for _ in range(B)]).astype(np.int32)
    pn = np.stack([rs.permutation(N) for _ in range(B)]).astype(np.int32)
    return props, cls, gt, pp, pn


@pytest.mark.gpu
@pytest.mark.parametrize("G", [4000, 8192])
def test_detection_targets_large_gt_shared_memory(_cuda, kernel_trace, G):
    """G > 3072 GT boxes: detection_iou_kernel keeps them in more than 48 KiB of dynamic shared memory (128 KiB at the
    8192 cap). Every index list, count, IoU and target bit-exact."""
    rs = np.random.RandomState(G)
    inputs = _many_gt_inputs(rs, 2, 2000, G)
    d, names = kernel_trace(lambda: _check_targets(Conf(), *inputs))
    assert_launched(names, must=["od::detection_iou_kernel(", "od::detection_target_kernel("])
    assert (d["counts"][:, 1] > 3072).all()                                        # valid GT boxes beyond 48 KiB
    n_pos = d["counts"][:, 4]
    assert (n_pos > 0).all()
    assert max(d["gt_assignment"][b, :n_pos[b]].max() for b in range(2)) > 3072


def _targets_with_masks(conf, props, cls, gt, pp, pn, masks, layout_hwg):
    """od_detection_target_forward with gt_masks in the [B,Mh,Mw,G] (layout_hwg = 1) or [B,G,Mh,Mw] layout."""
    from objectdetection_b200 import _lib
    B, N = props.shape[:2]
    G, R = cls.shape[1], conf.MRCNN_TRAIN_ROIS_PER_IMAGE
    mh, mw = conf.MASK_SHAPE
    t = {k: cu(v) for k, v in dict(props=props, cls=cls, gt=gt, pp=pp, pn=pn, masks=masks).items()}
    rois = torch.empty((B, R, 4), dtype=torch.float32, device="cuda")
    rcls = torch.empty((B, R), dtype=torch.int32, device="cuda")
    deltas = torch.empty((B, R, 4), dtype=torch.float32, device="cuda")
    targets = torch.full((B, R, mh, mw), -1.0, dtype=torch.float32, device="cuda")
    params = _lib.TargetParams(R, (ctypes.c_float * 4)(*conf.BBOX_STD_DEV), mh, mw, 1 if conf.USE_MINI_MASK else 0,
                               layout_hwg)
    L = _lib.lib()
    dl = _lib.DL()
    ws = _lib.workspace(L.od_detection_target_workspace_bytes(B, N, G), rois.device)
    _lib.check(L.od_detection_target_forward(dl(t["props"]), dl(t["cls"]), dl(t["gt"]), dl(t["pp"]), dl(t["pn"]),
                                             ctypes.byref(params), dl(rois), dl(rcls), dl(deltas), dl(t["masks"]),
                                             dl(targets), None, ws.data_ptr(), ws.numel(), _lib.stream_ptr(rois.device)),
               "od_detection_target_forward")
    return host(rois), host(targets)


@pytest.mark.gpu
@pytest.mark.parametrize("mini", [True, False])
def test_mask_targets_both_layouts_non_square(_cuda, kernel_trace, mini):
    """Mask targets of shape (28, 14) from non-square (48 x 40) GT masks, once in the reference's [B,Mh,Mw,G] layout
    and once in the [B,G,Mh,Mw] layout of the C ABI: both equal the oracle."""
    class C(Conf):
        USE_MINI_MASK = mini
        MASK_SHAPE = (28, 14)
    conf = C()
    rs = np.random.RandomState(13)
    B, N, G, Mh, Mw = 3, 600, 20, 48, 40
    props, cls, gt, pp, pn = _synth.target_inputs(rs, B, N, G, n_pad=100)
    masks = np.zeros((B, Mh, Mw, G), f32)
    yy, xx = np.mgrid[0:Mh, 0:Mw]
    for b in range(B):
        for g in range(G):
            cy, cx, ry, rx = rs.uniform(8, 40), rs.uniform(8, 32), rs.uniform(5, 22), rs.uniform(3, 12)
            masks[b, :, :, g] = (((yy - cy) / ry) ** 2 + ((xx - cx) / rx) ** 2 < 1).astype(f32)
    (rois1, got1), names = kernel_trace(lambda: _targets_with_masks(conf, props, cls, gt, pp, pn, masks, 1))
    assert_launched(names, must=["od::mask_target_kernel("])
    rois0, got0 = _targets_with_masks(conf, props, cls, gt, pp, pn, np.ascontiguousarray(masks.transpose(0, 3, 1, 2)), 0)
    assert np.array_equal(got0, got1) and np.array_equal(rois0, rois1)
    R = conf.MRCNN_TRAIN_ROIS_PER_IMAGE
    n_pos_total = 0
    for b in range(B):
        w_rois, _, _, wd = oracle.detection_targets(props[b], cls[b], gt[b], pp[b], pn[b], R, conf.BBOX_STD_DEV)
        assert_bits(rois1[b], w_rois, "rois")
        want = oracle.mask_targets(w_rois, cls[b], gt[b], masks[b], wd, (28, 14), mini)
        assert np.array_equal(got1[b], want), (b, np.abs(got1[b] - want).sum())
        n_pos_total += int(wd["counts"][4])
    assert n_pos_total > 0 and 0 < got1.mean() < 1


# ------------------------------------------------------------------ top-k
def _check_topk(s, k):
    from objectdetection_b200.proposals import top_k
    v, i = top_k(cu(s), k)
    wv, wi = oracle.topk(s, k)
    assert np.array_equal(host(i), wi)
    assert_bits(host(v), wv, "values")


@pytest.mark.gpu
def test_topk_one_cta_per_row(_cuda, kernel_trace):
    """rows >= 296 (two CTAs per SM over 148 SMs): the histogram and split passes run one CTA per row."""
    rs = np.random.RandomState(300)
    s = (np.round(rs.random_sample((300, 4092)) * 256) / 256).astype(f32)           # ties
    _, names = kernel_trace(lambda: _check_topk(s, 1000))
    assert_launched(names, must=["od::topk_hist1_kernel(", "od::topk_split_kernel(", "od::topk_tail_kernel(",
                                 "od::topk_merge_emit_kernel("], must_not=["od::topk_collect_kernel("])


@pytest.mark.gpu
@pytest.mark.parametrize("rows,cols,k,merge", [(2, 70000, 16384, True), (2, 70000, 16385, False),
                                               (2, 4092, 4091, True), (1, 20000, 19999, False)])
def test_topk_merge_and_global_sort_boundary(_cuda, kernel_trace, rows, cols, k, merge):
    """k = 16384 is the largest k of the tile sort + merge (128 KiB of dynamic shared memory); k = 16385 sorts the
    winners in global memory. k = cols - 1 leaves out exactly one score."""
    rs = np.random.RandomState(k)
    s = rs.random_sample((rows, cols)).astype(f32)
    s[0, ::7] = s[0, 3]                                                             # ties
    _, names = kernel_trace(lambda: _check_topk(s, k))
    merge_k = ["od::topk_tile_sort_kernel(", "od::topk_merge_emit_kernel("]
    sort_k = ["od::bitonic_step_global_kernel(", "od::pad_emit_kernel("]
    assert_launched(names, must=merge_k if merge else sort_k, must_not=sort_k if merge else merge_k)


# ------------------------------------------------------------------ RPN targets
@pytest.mark.gpu
@pytest.mark.parametrize("G", [256, 257])
def test_rpn_targets_fused_per_gt_boundary(_cuda, kernel_trace, G):
    """G <= 256: the anchor pass also finds each GT box's best anchor (rpn_gt_reduce_kernel combines the CTAs);
    G = 257: a separate per-GT pass (rpn_gt_best_kernel). Labels, counts and deltas against the oracle."""
    from objectdetection_b200.data_processor import PreprareTrainData

    class Sub(Conf):
        IMAGE_SHAPE = [256, 256, 3]
        RPN_ANCHOR_SCALES = (16, 32, 64, 128, 256)
    conf = Sub()
    P = PreprareTrainData(conf)
    anc = host(P.anchors)
    A, B, T = anc.shape[0], 2, conf.RPN_TRAIN_ANCHORS_PER_IMAGE
    rs = np.random.RandomState(G)
    cnt = np.array([G, G - 17], np.int32)
    gt = np.zeros((B, G, 4))
    for b in range(B):
        gt[b, :cnt[b]] = np.round(np.clip(anc[rs.choice(A, cnt[b], replace=False)] + rs.normal(0, 3, (cnt[b], 4)), 0, 256))
        bad = (gt[b, :, 2] <= gt[b, :, 0]) | (gt[b, :, 3] <= gt[b, :, 1])
        gt[b, bad] = [100, 100, 164, 164]
    pp = np.stack([rs.permutation(A) for _ in range(B)]).astype(np.int32)
    pn = np.stack([rs.permutation(A) for _ in range(B)]).astype(np.int32)
    out, names = kernel_trace(lambda: [host(x) for x in P.build_rpn_targets(gt, perm_pos=pp, perm_neg=pn, gt_count=cnt,
                                                                              return_counts=True)])
    pos, cls, bbox, counts = out
    fused = ["od::rpn_anchor_best_kernel<true>(", "od::rpn_gt_reduce_kernel("]
    per_gt = ["od::rpn_anchor_best_kernel<false>(", "od::rpn_gt_best_kernel("]
    assert_launched(names, must=fused if G <= 256 else per_gt, must_not=per_gt if G <= 256 else fused)
    for b in range(B):
        w_pos, w_cls, w_bbox, w_counts = oracle.rpn_targets(anc, gt[b, :cnt[b]], pp[b], pn[b], T, conf.RPN_BBOX_STDDEV)
        assert np.array_equal(counts[b], w_counts), (counts[b], w_counts)
        assert np.array_equal(cls[b], w_cls)
        n = w_counts[2]
        assert np.array_equal(pos[b, :n], w_pos) and not pos[b, n:].any()
        assert np.allclose(bbox[b], w_bbox, rtol=1e-13, atol=0)
    assert (counts[:, 2] == T // 2).all()                   # more positives than targets: subsampled through perm_pos


# ------------------------------------------------------------------ past the caps
def _refused(trace, fn):
    """fn must raise ValueError without launching any of the library's kernels. A torch kernel runs first so that the
    trace is known to record kernels."""
    def run():
        torch.ones(1, device="cuda").add_(1)
        with pytest.raises(ValueError) as e:
            fn()
        return e
    e, names = trace(run)
    assert_launched(names, must_not=["od::"])
    return str(e.value)


@pytest.mark.gpu
def test_past_the_caps_refused_before_any_launch(_cuda, kernel_trace):
    """DetectionLayer N = 16385, DetectionTargetLayer G = 8193 and roi_processing_order with 4097 ROIs per image are
    one past the advertised caps: OD_ERR_PARAM (ValueError) before any kernel of the library runs."""
    from objectdetection_b200 import BuildDetectionTargets, DetectionLayer
    from objectdetection_b200.maskrcnn import roi_processing_order
    rs = np.random.RandomState(0)
    N = 16385
    props = cu(_synth.rois_log_uniform(rs, 1, N))
    probs, bbox = (cu(x) for x in _synth.head_outputs(rs, 1, N, 3))
    msg = _refused(kernel_trace, lambda: DetectionLayer(Conf(), [1024, 1024, 3], 1, WIN[:1], props, probs, bbox))
    assert "16384" in msg
    p, c, g, pp, pn = (cu(x) for x in _many_gt_inputs(rs, 1, 300, 8193, n_pad=20))
    msg = _refused(kernel_trace, lambda: BuildDetectionTargets(ShapesConfig(), p, c, g, perm_pos=pp, perm_neg=pn))
    assert "8192" in msg
    rois = cu(_synth.rois_log_uniform(rs, 2, 4097))
    msg = _refused(kernel_trace, lambda: roi_processing_order(rois, [1024, 1024, 3]))
    assert "4096" in msg
