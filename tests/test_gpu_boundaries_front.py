"""Size boundaries of the proposal front, of Faster R-CNN roi_pool and of the bfloat16 kernel overloads, run on both
sides through the C ABI against the CPU oracle, with the machinery of test_gpu_boundaries.py: a Boundary table whose
values come from Python restatements of the planning code, sentinel-filled outputs, a workspace poisoned with 0xFF bytes,
bit-for-bit comparison (padding included), the "no sentinel survives" check and, where the kernels change, the trace.

The rows cover:
- od_frcnn_proposal_forward: the end of the staged NMS scan (Faster R-CNN calls nms_scan_launch directly: one round, no
  wide scan, so past the ring it runs the unstaged nms_scan_kernel<false>), the rank sort's 1024-key tile and 32-key CTA,
  the mask kernel's 64-box tiles, the emit kernel's last CTA and its offset reduction over B > 256 images, and
  K = min(total, pre_n);
- od_proposal_forward / _levels: K against A, N against K, the last CTA of the decode and gather grids, and the level
  search of the per-level tables (top scores on both sides of every level's first anchor, a 1x1 level, 1 and 8 levels);
- od_roi_pool_forward: the last CTA of crop_pool_bins_kernel (kPoolBins pooled bins each) at thin and wide depths;
- the bf16 overloads of ROIAlign (crop_rows grid, mask branch, order pre-pass, the tier edge and the last CTA of both
  flat kernels at bf16 unit sizes), DetectionLayer and the head losses, on the edges of test_gpu_boundaries.py's rows.

bf16 rows check the contract of DESIGN.md section 2: a bf16 input is widened exactly, so an fp32 result equals the fp32
path and the oracle on the widened inputs bit for bit, and a bf16 result is the round-to-nearest-even of that fp32 value
(torch's float32 -> bfloat16 conversion). The trace must show the bf16 overload, never the fp32 kernel.

test_front_constants_match_sources and test_front_table_values need no GPU: they read the constants, the MapUnit channel
counts and the literal thresholds restated here from objectdetection_b200/csrc and fail when the sources move."""
import ctypes
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
from test_gpu_boundaries import (BF16, BY_NAME as BASE_ROWS, CSRC, F32, NMS_STAGED_LIMIT, Boundary, _L, _edge_rois,  # noqa: E402
                                 _roi_maps, assert_written, bf16_round, check_sources, nms_slots, poison, resolve,
                                 run_detection, run_mrcnn_loss, run_rpn_loss, sent_f32, sent_i32)
from test_gpu_dispatch import _assert_close_f64, _cuda, assert_launched, kernel_trace  # noqa: E402,F401
from test_gpu_parity import assert_bits, cu, host  # noqa: E402

torch = pytest.importorskip("torch")
f32, f64 = np.float32, np.float64
B_SENT = 0x7FBD                                                                 # bf16 sentinel (a NaN no kernel writes)

# ------------------------------------------------------------------ constants of the planning code
CONST = {
    "kFrRankThreads": ("frcnn.cu", 256),
    "kFrRankMine": ("frcnn.cu", 32),
    "kFrRankTile": ("frcnn.cu", 1024),
    "kFrEmitThreads": ("frcnn.cu", 256),
    "kPoolBins": ("roi_align.cu", 32),
    "kBinBins": ("roi_align.cu", 32),
    "kBinThreads": ("roi_align.cu", 128),
    "kRowsD4": ("roi_align.cu", 64),
    "kRowsPixelBytes": ("roi_align.cu", 1024),
}
# channels per 16-byte map unit, `static constexpr int kCh` of MapUnit<TMap> (roi_align.cu)
MAP_UNIT_CH = {"float": 4, "__nv_bfloat16": 8}
LITERALS = [
    ("frcnn.cu", "const int64_t K = total < params->pre_nms_top_n ? total : params->pre_nms_top_n;"),
    ("frcnn.cu", "const dim3 grid((unsigned)((total + kFrRankMine - 1) / kFrRankMine), (unsigned)B);"),
    ("frcnn.cu", "for (int64_t t0 = 0; t0 < total; t0 += kFrRankTile) {"),
    ("frcnn.cu", "const dim3 grid((unsigned)W, (unsigned)W, (unsigned)B);"),
    ("frcnn.cu", "frcnn_mask_kernel<<<grid, 64, 0, st>>>"),
    # one round, no wide scan (wide = nullptr): past the ring the unstaged scan
    ("frcnn.cu", "OD_CHECK(nms_scan_launch(f.mask, f.diagT, npre, B, K, nms_mask_stride(K), post_n, f.keep_pos, num_kept, "
                 "nullptr, st));"),
    ("nms.cu", "return scan_round_launch(mask, diagT, num_valid, B, K, mask_stride, max_out, 0, W, 1, nullptr, keep_pos, "
               "num_kept, keep_flag, nullptr, st);"),
    ("nms.cu", "plain + 2 * per_slot <= kSmemBudget"),
    ("frcnn.cu", "const dim3 egrid((unsigned)((post_n + kFrEmitThreads - 1) / kFrEmitThreads), (unsigned)B);"),
    ("frcnn.cu", "for (int q = threadIdx.x; q < B; q += kFrEmitThreads) {"),
    ("proposal.cu", "const int64_t K = params->pre_nms_limit < A ? params->pre_nms_limit : A;"),
    ("proposal.cu", "const dim3 grid((unsigned)((total + 255) / 256));"),
    ("proposal.cu", "launch_pdl(proposal_gather_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256)"),
    ("proposal.cu", "while (l + 1 < t.num_levels && i >= t.off[l + 1]) ++l;"),
    ("proposal.cu", "proposals[t] = (p >= 0) ? clipped[b * K + p] : make_float4(0.f, 0.f, 0.f, 0.f);"),
    ("../../include/odhead.h", "#define OD_MAX_LEVELS 8"),
    ("roi_align.cu", "const int64_t total_bins = n * 49;"),
    ("roi_align.cu", "const int64_t grid = (total_bins + kPoolBins - 1) / kPoolBins;"),
    ("roi_align.cu", "const int32_t D4 = D / MapUnit<TMap>::kCh;"),
    ("roi_align.cu", "if (lg >= 0 && D4 >= 16) {"),
    ("roi_align.cu", "constexpr int BINS = 512;"),
    ("roi_align.cu", "template <typename TMap> constexpr int kRowsUnits = 4 * kRowsD4 / MapUnit<TMap>::kCh;"),
    ("roi_align.cu", "if (D != 4 * kRowsD4 || ph > kRowsMaxPool || pw > kRowsMaxWidth || pmax < kRowsMinPool"),
    ("roi_align.cu", "const int64_t grid = n_rois < (int64_t)sms[dev] ? n_rois : (int64_t)sms[dev];"),
    ("roi_align.cu", "n_rois >= 512 && src.rois_per_image <= kOrderThreads * kOrderPerThread"),
]
OD_MAX_LEVELS = 8


def C(name):
    return CONST[name][1]


def parse_map_units(csrc=CSRC):
    src = open(os.path.join(csrc, "roi_align.cu")).read()
    return {t: int(n) for t, n in re.findall(r"struct\s+MapUnit<([\w:]+)>\s*\{[^}]*?kCh\s*=\s*(\d+)\s*;", src)}


# ------------------------------------------------------------------ the planning formulas, restated
TNAME = {F32: "float", BF16: "__nv_bfloat16"}


def units(D, map_dt):
    """launch_crop_bins: 16-byte units per pixel, D / MapUnit<TMap>::kCh."""
    return D // MAP_UNIT_CH[TNAME[map_dt]]


def bins_tier(D, map_dt):
    """The crop_bins CTA size (bins): kBinBins for a power-of-two unit count >= 16, else 512."""
    u = units(D, map_dt)
    return C("kBinBins") if u & (u - 1) == 0 and u >= 16 else 512


def rows_units(map_dt):
    """kRowsUnits<TMap>: 16-byte units of a D = 4 kRowsD4 pixel (one per lane and 32 lanes, or two)."""
    return 4 * C("kRowsD4") // MAP_UNIT_CH[TNAME[map_dt]]


def frcnn_scan(K):
    """od_frcnn_proposal_forward's keep scan: one round of nms_scan_launch without the wide scan."""
    return "od::nms_scan_kernel<true>(" if nms_slots(K) >= 2 else "od::nms_scan_kernel<false>("


def cdiv(a, b):
    return (a + b - 1) // b


# ------------------------------------------------------------------ the table
def vid(v):
    return "-".join(map(str, v)) if isinstance(v, tuple) else str(v)


PAIRS = [(BF16, F32), (F32, BF16), (BF16, BF16)]
PAIR_ID = {(BF16, F32): "bf16>f32", (F32, BF16): "f32>bf16", (BF16, BF16): "bf16>bf16", (F32, F32): "f32>f32"}
BY_PAIR_ID = {v: k for k, v in PAIR_ID.items()}
HEAD_PAIR_ID = {(BF16, F32): "bf16+f32", (F32, BF16): "f32+bf16", (BF16, BF16): "bf16+bf16", (F32, F32): "f32+f32"}
BY_HEAD_PAIR_ID = {v: k for k, v in HEAD_PAIR_ID.items()}
FRCNN_TOTAL = 38 * 63 * 9                                                      # 600x1000 at stride 16, 9 anchors
RANK_TILE, RANK_MINE, EMIT = C("kFrRankTile"), C("kFrRankMine"), C("kFrEmitThreads")
A_PROP, K_PROP = 1000, 500


def _crop_kernels(v, sms, pool, D):
    """ROIAlign kernels of a bf16 dtype pair: the named overload, never the fp32 kernel."""
    md, od = BY_PAIR_ID[v[0]]
    m, o = TNAME[md], TNAME[od]
    if pool == (14, 14) and D == 4 * C("kRowsD4"):
        must = [f"od::crop_rows_kernel<{m},{o}>("]
    else:
        must = [f"od::crop_bins_kernel<{m},{o},{bins_tier(D, md)},2,true,false>("]
    return must, ["od::crop_rows_kernel(", "od::crop_bins_kernel<32,", "od::crop_bins_kernel<512,"]


def _pyr_kernels(v, sms):
    md, od = BY_PAIR_ID[v[0]]
    m, o = TNAME[md], TNAME[od]
    must = [f"od::crop_rows_kernel<{m},{o}>("]
    must_not = ["od::crop_rows_kernel(", "od::crop_bins_kernel<"]
    if v[1] >= 512:
        must.append("od::roi_order_kernel(")
    else:
        must_not.append("od::roi_order_kernel(")
    return must, must_not


def _head_kernels(kind):
    def k(v, sms):
        a, b = (TNAME[t] for t in BY_HEAD_PAIR_ID[v[0]])
        if kind == "det":
            return [f"od::det_prepare_kernel<{a},{b}>("], ["od::det_prepare_kernel("]
        if kind == "mrcnn":
            return [f"od::mrcnn_loss_kernel<{a},{b}>("], ["od::mrcnn_loss_kernel("]
        names = [f"od::rpn_loss_class_kernel{'<__nv_bfloat16>' if a != 'float' else ''}(",
                 f"od::rpn_loss_box_kernel{'<__nv_bfloat16>' if b != 'float' else ''}("]
        other = [f"od::rpn_loss_class_kernel{'<__nv_bfloat16>' if a == 'float' else ''}(",
                 f"od::rpn_loss_box_kernel{'<__nv_bfloat16>' if b == 'float' else ''}("]
        return names, other
    return k


def _prop_kernels(v, sms):
    bf = v[0] == "bf16"
    dec = "od::proposal_decode_kernel<__nv_bfloat16,false>(" if bf else "od::proposal_decode_kernel<false>("
    other = "od::proposal_decode_kernel<false>(" if bf else "od::proposal_decode_kernel<__nv_bfloat16,"
    return [dec, "od::proposal_gather_kernel("], [other, "od::rpn_level_scores_kernel"]


def _levels_kernels(v, sms):
    lg, bb = (t == "bf16" for t in v[1].split("+"))
    must = ["od::rpn_level_scores_kernel<__nv_bfloat16>(" if lg else "od::rpn_level_scores_kernel(",
            "od::proposal_decode_kernel<__nv_bfloat16,true>(" if bb else "od::proposal_decode_kernel<true>("]
    must_not = ["od::rpn_level_scores_kernel(" if lg else "od::rpn_level_scores_kernel<",
                "od::proposal_decode_kernel<true>(" if bb else "od::proposal_decode_kernel<__nv_bfloat16,"]
    return must, must_not


LEVEL_SETS = {
    "L1": [(9, 7)],
    "L5": [(8, 6), (4, 4), (2, 3), (1, 1), (3, 2)],                             # a 1x1 level between two others
    "L8": [(6, 5), (4, 4), (1, 1), (3, 3), (2, 3), (2, 2), (1, 2), (1, 1)],     # OD_MAX_LEVELS levels
}
LEVEL_PAIRS = ["f32+f32", "bf16+bf16", "bf16+f32", "f32+bf16"]
_grid_edge = 256                                                                # decode / gather CTAs of 256 threads

BOUNDARIES = [
    Boundary("frcnn_staged_limit", "od_frcnn_proposal_forward", "pre_nms_top_n (38x63x9, post_n = pre_n, fp32)",
             [NMS_STAGED_LIMIT - 1, NMS_STAGED_LIMIT],
             "scan_round_launch: plain + 2 * per_slot <= 200 KiB; Faster R-CNN has no wide scan, so past it the "
             "single-round unstaged scan",
             kernels=lambda v, sms: ([frcnn_scan(v), "od::frcnn_mask_kernel("],
                                     ["od::nms_scan_wide_kernel<"] + [k for k in ("od::nms_scan_kernel<true>(",
                                                                                   "od::nms_scan_kernel<false>(")
                                                                      if k != frcnn_scan(v)])),
    Boundary("frcnn_rank_tile", "od_frcnn_proposal_forward", "total anchors (fp64, 1 anchor, fh = 1, pre_n = total)",
             [RANK_TILE - 1, RANK_TILE, RANK_TILE + 1, 2 * RANK_TILE - 1, 2 * RANK_TILE + 1],
             "frcnn_rank_gather_kernel: kFrRankTile keys per shared tile (zero-filled tail), kFrRankMine keys per CTA",
             kernels=lambda v, sms: (["od::frcnn_rank_gather_kernel("], ["od::frcnn_gather_kernel(", "od::topk_"])),
    Boundary("frcnn_mask_tile", "od_frcnn_proposal_forward", "npre = pre_n < valid boxes (fp32, fp64)",
             [(dt, n) for dt in ("f32", "f64") for n in (63, 64, 65, 127, 128, 129)],
             "frcnn_mask_kernel: 64x64-box tiles, the diagonal tile transposed, the last tile partial",
             kernels=lambda v, sms: (["od::frcnn_mask_kernel(", "od::frcnn_gather_kernel(" if v[0] == "f32" else
                                      "od::frcnn_rank_gather_kernel("], [])),
    Boundary("frcnn_emit", "od_frcnn_proposal_forward", "(B, post_n), fp32",
             [(2, EMIT - 1), (2, EMIT), (2, EMIT + 1), (EMIT, 20), (EMIT + 1, 20)],
             "frcnn_emit_kernel: ceil(post_n / kFrEmitThreads) CTAs; the per-image offsets reduce num_kept over B in "
             "strides of kFrEmitThreads; rows from the batch's total on are zeroed",
             kernels=lambda v, sms: (["od::frcnn_emit_kernel("], [])),
    Boundary("frcnn_pre_vs_total", "od_frcnn_proposal_forward", "pre_n (7x9x9 = 567 anchors), fp32 and fp64",
             [(dt, 567 + d) for dt in ("f32", "f64") for d in (-1, 0, 1)],
             "od_frcnn_proposal_forward: K = min(total, pre_nms_top_n); rows past the kept ones are zero"),
    Boundary("proposal_k_vs_a", "od_proposal_forward", f"pre_nms_limit (A = {A_PROP}), fp32 and bf16 deltas",
             [(dt, A_PROP + d) for dt in ("f32", "bf16") for d in (-1, 0, 1)],
             "proposal_core: K = min(pre_nms_limit, A); top-k with k = cols, the decode reads ix",
             kernels=_prop_kernels),
    Boundary("proposal_n_vs_k", "od_proposal_forward", f"post_nms_count (K = {K_PROP}), fp32 and bf16 deltas",
             [(dt, K_PROP + d) for dt in ("f32", "bf16") for d in (-1, 0, 1)],
             "proposal_gather_kernel: keep_pos -1 rows are zero padding", kernels=_prop_kernels),
    Boundary("proposal_grids", "od_proposal_forward", "B*K = B*N (B = 1), fp32 and bf16 deltas",
             [(dt, _grid_edge + d) for dt in ("f32", "bf16") for d in (-1, 0, 1)],
             "proposal_decode_kernel / proposal_gather_kernel: ceil(total / 256) CTAs of 256 threads",
             kernels=_prop_kernels),
    Boundary("levels_edges", "od_proposal_forward_levels", "level tables (logits + deltas dtypes)",
             [(s, p) for s in LEVEL_SETS for p in LEVEL_PAIRS],
             "level_row: the level of anchor i is the last l with i >= off[l]; top scores at off[l] - 1 and off[l]",
             kernels=_levels_kernels),
    Boundary("roi_pool_bins", "od_roi_pool_forward", "(n, D)", [(n, D) for D in (4, 8, 512) for n in (1, 31, 32, 33)],
             "crop_pool_bins_kernel: kPoolBins pooled bins per CTA over 49 n bins",
             kernels=lambda v, sms: (["od::crop_pool_bins_kernel("], [])),
    Boundary("bf16_crop_rows_grid", "od_crop_and_resize", "n_rois (14x14, D = 256), (maps > pooled)",
             [(PAIR_ID[p], n) for p in PAIRS for n in (1, "sms-1", "sms", "sms+1")],
             "launch_crop_rows: grid = min(n_rois, runtime SMs); kRowsUnits<TMap> units per pixel",
             kernels=lambda v, sms: _crop_kernels(v, sms, (14, 14), 256)),
    Boundary("bf16_mask_branch", "od_pyramid_roi_align_forward_ws", "B*N (B = 1, 14x14, D = 256, ticket workspace)",
             [(PAIR_ID[p], n) for p in PAIRS for n in (1, 100)],
             "the mask branch pools <= 100 detections of an image", kernels=_pyr_kernels),
    Boundary("bf16_roi_order", "od_pyramid_roi_align_forward_ws / _ordered", "n_rois (B = 1, 14x14, D = 256)",
             [(PAIR_ID[p], n) for p in PAIRS for n in (511, 512)],
             "launch_crop_bins: the order pre-pass needs n_rois >= 512; _ordered takes the caller's order",
             kernels=_pyr_kernels),
    Boundary("bf16_tier", "od_crop_and_resize", "D (1x1 crops, 40 ROIs)", [(PAIR_ID[p], D) for p in PAIRS for D in (64, 128)],
             "launch_crop_bins: kBinBins tier iff D / kCh is a power of two >= 16 (D = 128 for bf16 maps, 64 for fp32)",
             kernels=lambda v, sms: _crop_kernels(v, sms, (1, 1), v[1])),
    Boundary("bf16_bins_32", "od_crop_and_resize", "total_bins (1x1 crops, D = 128)",
             [(PAIR_ID[p], n) for p in PAIRS for n in sorted({2 * C("kBinBins") + d for d in (-1, 0, 1)})],
             "crop_bins_kernel<kBinBins>: the last CTA's bins at 16 bf16 units per pixel",
             kernels=lambda v, sms: _crop_kernels(v, sms, (1, 1), 128)),
    Boundary("bf16_bins_512", "od_crop_and_resize", "total_bins (1x1 crops, D = 8: one bf16 unit)",
             [(PAIR_ID[p], n) for p in PAIRS for n in (511, 512, 513)],
             "crop_bins_kernel<BINS = 512>: the last CTA's bins",
             kernels=lambda v, sms: _crop_kernels(v, sms, (1, 1), 8)),
    Boundary("bf16_det", "od_detection_forward", "det_rank_tile, det_rank_vs_sort, det_finalize_kept values",
             [(HEAD_PAIR_ID[p], r, v) for p in PAIRS for r in ("det_rank_tile", "det_rank_vs_sort", "det_finalize_kept")
              for v in BASE_ROWS[r].values],
             "the rows of test_gpu_boundaries.py with bf16 mrcnn_class_probs and / or mrcnn_bbox",
             kernels=_head_kernels("det")),
    Boundary("bf16_rpn_loss", "od_rpn_loss_forward", "rpn_loss_chunk values",
             [(HEAD_PAIR_ID[p], v) for p in PAIRS for v in BASE_ROWS["rpn_loss_chunk"].values],
             "rpn_loss_class_kernel / rpn_loss_box_kernel bf16 overloads: kLossChunk anchors per CTA",
             kernels=_head_kernels("rpn")),
    Boundary("bf16_mrcnn_loss", "od_mrcnn_loss_forward", "mrcnn_loss_cta values",
             [(HEAD_PAIR_ID[p], v) for p in PAIRS for v in BASE_ROWS["mrcnn_loss_cta"].values],
             "mrcnn_loss_kernel<TL, TB>: one 1024-thread CTA loops over B*R", kernels=_head_kernels("mrcnn")),
]
BY_NAME = {b.name: b for b in BOUNDARIES}
CASES = [pytest.param(b.name, v, id=f"{b.name}-{vid(v)}") for b in BOUNDARIES for v in b.values]


# ------------------------------------------------------------------ no GPU: the table follows the sources
def test_front_constants_match_sources():
    check_sources(CONST, LITERALS)
    assert parse_map_units() == MAP_UNIT_CH, f"MapUnit channel counts changed: {parse_map_units()}; update MAP_UNIT_CH"


def test_front_table_values():
    """The restated formulas change exactly at the table's values."""
    assert NMS_STAGED_LIMIT == 12545 < FRCNN_TOTAL
    assert frcnn_scan(NMS_STAGED_LIMIT - 1) == "od::nms_scan_kernel<true>("
    assert frcnn_scan(NMS_STAGED_LIMIT) == "od::nms_scan_kernel<false>("
    assert [cdiv(t, RANK_TILE) for t in BY_NAME["frcnn_rank_tile"].values] == [1, 1, 2, 2, 3]
    assert [t % RANK_MINE for t in BY_NAME["frcnn_rank_tile"].values] == [31, 0, 1, 31, 1]
    assert [cdiv(n, 64) for _, n in BY_NAME["frcnn_mask_tile"].values[:6]] == [1, 1, 2, 2, 2, 3]
    assert [cdiv(p, EMIT) for _, p in BY_NAME["frcnn_emit"].values[:3]] == [1, 1, 2]
    assert [B > EMIT for B, _ in BY_NAME["frcnn_emit"].values] == [False, False, False, False, True]
    assert [cdiv(v, 256) for _, v in BY_NAME["proposal_grids"].values[:3]] == [1, 1, 2]
    assert [cdiv(49 * n, C("kPoolBins")) for n, _ in BY_NAME["roi_pool_bins"].values[:4]] == [2, 48, 49, 51]
    assert [49 * n % C("kPoolBins") for n, _ in BY_NAME["roi_pool_bins"].values[:4]] == [17, 15, 0, 17]
    assert units(8, BF16) == 1 and units(8, F32) == 2
    assert bins_tier(64, BF16) == 512 and bins_tier(128, BF16) == 32 and bins_tier(64, F32) == 32
    assert rows_units(F32) == 64 and rows_units(BF16) == 32
    assert 16 * rows_units(F32) == C("kRowsPixelBytes") == 2 * 16 * rows_units(BF16)
    assert max(len(s) for s in LEVEL_SETS.values()) == OD_MAX_LEVELS and any((1, 1) in s for s in LEVEL_SETS.values())
    for b in BOUNDARIES:
        assert len(b.values) >= 2 and len(set(map(vid, b.values))) == len(b.values), b.name
        assert b.source and b.entry.startswith("od_"), b.name


# ------------------------------------------------------------------ GPU helpers
def sent_bf16(shape):
    return torch.full(shape, B_SENT, dtype=torch.int16, device="cuda").view(BF16)


def sent_out(shape, dt):
    return sent_bf16(shape) if dt == BF16 else sent_f32(shape)


def assert_written16(t, what, untouched=None):
    """bf16 output: no sentinel half-word outside `untouched` rows, every one inside them untouched."""
    h = host(t.view(torch.int16)).view(np.uint16)
    hit = (h == B_SENT).reshape(h.shape[0], -1)
    if untouched is None:
        untouched = np.zeros(h.shape[0], bool)
    bad = np.argwhere(hit & ~untouched[:, None])
    assert bad.size == 0, f"{what}: {bad.shape[0]} bf16 words still hold the sentinel, first at {bad[:3].tolist()}"
    assert hit[untouched].all(), f"{what}: rows that must stay untouched were written"


def check_out(t, want32, dt, what, untouched=None):
    """An output of dtype dt against the fp32 reference want32: bit for bit, after rounding to bf16 for a bf16 output;
    rows in `untouched` are only checked to be untouched."""
    keep = np.ones(want32.shape[0], bool) if untouched is None else ~untouched
    got = host(t.float())
    want = bf16_round(want32) if dt == BF16 else want32
    assert_bits(got[keep], want[keep], what)
    if dt == BF16:
        assert_written16(t, what, untouched)
    else:
        assert_written(got, what, untouched)
    return got


# ------------------------------------------------------------------ Faster R-CNN proposals
def _frcnn_params(pre_n, post_n, na, image_h, image_w, stride, min_hw, thr, base):
    from objectdetection_b200 import _lib
    p = _lib.FrcnnParams()
    p.feat_stride, p.image_h, p.image_w, p.min_box_hw = stride, image_h, image_w, min_hw
    p.pre_nms_top_n, p.post_nms_top_n, p.nms_threshold, p.num_anchors = pre_n, post_n, thr, na
    for i, v in enumerate(np.asarray(base, f64).reshape(-1)):
        p.base_anchors[i] = float(v)
    return p


def _frcnn_inputs(rs, B, fh, fw, na, sd=0.5, small=0.1, dtype=f32):
    """Scores on a 1/512 grid (ties, resolved by index), deltas N(0, sd); a fraction `small` of the boxes shrunk below
    the 16 px minimum (filtered out, so their keys sort below every valid one)."""
    probs = np.round(rs.random_sample((B, fh, fw, 2 * na)) * 512) / 512
    bbox = rs.normal(0, sd, size=(B, fh, fw, 4 * na))
    d = bbox.reshape(B, -1, 4)
    d[rs.random_sample(d.shape[:2]) < small, 2:] = -8.0
    return probs.astype(dtype), bbox.astype(dtype)


SQUARE32 = np.array([[-8., -8., 23., 23.]])                                       # one 32 px anchor
SQUARE64 = np.array([[-24., -24., 39., 39.]])                                     # one 64 px anchor: neighbours overlap


def run_frcnn(trace, probs, bbox, pre_n, post_n, image_h, image_w, stride=16, min_hw=16, thr=0.7,
              base=oracle.FRCNN_BASE_ANCHORS):
    """od_frcnn_proposal_forward with sentinel outputs and a poisoned workspace against oracle.frcnn_proposals per image
    (column 0 = b), padding rows included. Returns the kernel names and the per-image counts."""
    _lib, L, dl = _L()
    B, fh, fw = probs.shape[:3]
    na = probs.shape[3] // 2
    base = np.asarray(base, f64)[:na]
    p = _frcnn_params(pre_n, post_n, na, image_h, image_w, stride, min_hw, thr, base)
    tp, tb = cu(probs), cu(bbox)
    props, num = sent_f32((B * post_n, 5)), sent_i32((B,))

    def call():
        ws = poison(L.od_frcnn_proposal_workspace_bytes_batch(B, fh, fw, ctypes.byref(p)), tp.device)
        _lib.check(L.od_frcnn_proposal_forward(dl(tp), dl(tb), ctypes.byref(p), dl(props), dl(num), ws.data_ptr(),
                                               ws.numel(), _lib.stream_ptr(tp.device)), "od_frcnn_proposal_forward")
    _, names = trace(call)
    got, gnum = host(props), host(num)
    want = np.zeros((B * post_n, 5), f32)
    counts, off = [], 0
    for b in range(B):
        r = oracle.frcnn_proposals(probs[b:b + 1].astype(f64), bbox[b:b + 1].astype(f64), image_h, image_w, pre_n, post_n,
                                   thr, min_hw=min_hw, feat_stride=stride, base_anchors=base)
        r[:, 0] = b
        want[off:off + r.shape[0]] = r
        off += r.shape[0]
        counts.append(r.shape[0])
    assert np.array_equal(gnum, counts), (gnum, counts)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), \
        f"proposals differ (padding included) in rows {np.unique(np.argwhere(got.view(np.uint32) != want.view(np.uint32))[:, 0])[:8]}"
    assert_written(got, "proposals")
    assert_written(gnum, "num_out")
    return names, np.array(counts)


def frcnn_case(trace, name, v):
    if name == "frcnn_staged_limit":
        rs = np.random.RandomState(v)
        probs, bbox = _frcnn_inputs(rs, 1, 38, 63, 9, small=0.0)
        names, counts = run_frcnn(trace, probs, bbox, v, v, 600, 1000, min_hw=1)      # every box valid: npre = pre_n
        assert counts[0] > 1000, counts
    elif name == "frcnn_rank_tile":
        rs = np.random.RandomState(v)
        probs, bbox = _frcnn_inputs(rs, 1, 1, v, 1, dtype=f64)
        probs[0, 0, -3:, 0] = probs.max()                                      # ties at the top, in the last CTA
        names, counts = run_frcnn(trace, probs, bbox, v, v, 64, 8 * v, stride=8, base=SQUARE32)
        assert counts[0] > 100, counts
    elif name == "frcnn_mask_tile":
        dt, n = v
        rs = np.random.RandomState(n)
        probs, bbox = _frcnn_inputs(rs, 2, 16, 20, 1, sd=0.3, dtype=f32 if dt == "f32" else f64)
        names, counts = run_frcnn(trace, probs, bbox, n, n, 256, 320, thr=0.5, base=SQUARE64)
        assert (counts < n).any() and (counts > 0).all(), counts                        # some boxes suppressed
    elif name == "frcnn_emit":
        B, post_n = v
        rs = np.random.RandomState(B * 1000 + post_n)
        side = 24 if B == 2 else 6
        probs, bbox = _frcnn_inputs(rs, B, side, side, 1, sd=0.2, small=0.0)
        d = bbox.reshape(B, -1, 4)
        if B == 2:
            d[1, 100:, 2:] = -8.0                                              # image 1: 100 valid boxes < post_n
        else:
            d[3:B - 1:7, :, 2:] = -8.0                                         # empty images inside the batch
            d[-1, 5:, 2:] = -8.0                                               # the last image keeps 5 < post_n
        names, counts = run_frcnn(trace, probs, bbox, side * side, post_n, 16 * side, 16 * side, base=SQUARE32)
        if B == 2:
            assert counts[0] >= post_n and counts[1] < post_n, counts
        else:
            assert (counts[3:B - 1:7] == 0).all() and 0 < counts[-1] < post_n and (counts[:3] == post_n).all(), counts
    elif name == "frcnn_pre_vs_total":
        dt, pre_n = v
        rs = np.random.RandomState(pre_n)
        probs, bbox = _frcnn_inputs(rs, 2, 7, 9, 9, dtype=f32 if dt == "f32" else f64)
        names, counts = run_frcnn(trace, probs, bbox, pre_n, 600, 112, 144)
    return names


# ------------------------------------------------------------------ Mask R-CNN proposals
STD = np.array([0.1, 0.1, 0.2, 0.2], f32)


def _prop_params(pre, post, thr=0.7):
    from objectdetection_b200 import _lib
    return _lib.ProposalParams((ctypes.c_float * 4)(*STD), pre, post, thr)


def _prop_debug(dl, B, K, N):
    """Sentinel-filled DEBUG outputs ix, scores, keep_idx and num_kept, and the od_proposal_debug pointing at them."""
    from objectdetection_b200 import _lib
    d = dict(ix=sent_i32((B, K)), scores=sent_f32((B, K)), keep_idx=sent_i32((B, N)), num_kept=sent_i32((B,)))
    dbg = _lib.ProposalDebug()
    for k, t in d.items():
        setattr(dbg, k, dl(t))
    return d, dbg


def _check_prop(got, d, want, wd, K):
    got = host(got)
    assert np.array_equal(host(d["ix"]), wd["ix"]), "ix"
    assert_bits(host(d["scores"]), wd["scores"], "scores")
    assert np.array_equal(host(d["num_kept"]), wd["num_kept"]), (host(d["num_kept"]), wd["num_kept"])
    assert np.array_equal(host(d["keep_idx"]), wd["keep_idx"]), "keep_idx (-1 padding included)"
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), "proposals (zero padding included)"
    assert_written(got, "proposals")
    for k, t in d.items():
        assert_written(host(t), k)
    return got


def _prop_inputs(rs, B, A):
    fg = (np.round(rs.random_sample((B, A)) * 256) / 256).astype(f32)           # ties
    probs = np.stack([1 - fg, fg], 2).astype(f32)
    anchors = _synth.rois_log_uniform(rs, B, A, lo=8, hi=200).astype(f32)
    bbox = rs.normal(0, 1, (B, A, 4)).astype(f32)
    return probs, bbox, anchors


def run_proposals(trace, dt, B, A, pre, post):
    _lib, L, dl = _L()
    rs = np.random.RandomState(A * 7 + pre + 3 * post)
    probs, bbox, anchors = _prop_inputs(rs, B, A)
    if dt == "bf16":
        bbox = bf16_round(bbox)
    K = min(pre, A)
    tp, tb, ta = cu(probs), cu(bbox).to(BF16 if dt == "bf16" else F32), cu(anchors)
    out = sent_f32((B, post, 4))
    d, dbg = _prop_debug(dl, B, K, post)
    params = _prop_params(pre, post)

    def call():
        ws = poison(L.od_proposal_workspace_bytes(B, A, ctypes.byref(params)), tp.device)
        _lib.check(L.od_proposal_forward(dl(tp), dl(tb), dl(ta), None, ctypes.byref(params), dl(out), ctypes.byref(dbg),
                                         ws.data_ptr(), ws.numel(), _lib.stream_ptr(tp.device)), "od_proposal_forward")
    _, names = trace(call)
    want, wd = oracle.proposal_forward(probs, bbox, anchors, STD, pre, post, 0.7, debug=True)
    _check_prop(out, d, want, wd, K)
    return names, wd


def _level_tensors(rs, B, shapes, a):
    lg = [rs.normal(0, 1.0, (B, h, w, 2 * a)).astype(f32) for h, w in shapes]
    bb = [rs.normal(0, 1, (B, h, w, 4 * a)).astype(f32) for h, w in shapes]
    off = np.cumsum([0] + [h * w * a for h, w in shapes])
    top = sorted({i for l in range(len(shapes)) for i in (off[l] - 1, off[l]) if 0 <= i < off[-1]} | {off[-1] - 1})
    for b in range(B):
        for r, i in enumerate(top):                                          # the highest scores, distinct, at the edges
            l = int(np.searchsorted(off, i, side="right") - 1)
            pair = lg[l].reshape(B, -1, 2)
            pair[b, i - off[l]] = [-6.0, 6.0 - 0.25 * r + 0.125 * b]
    return lg, bb, top, int(off[-1])


def run_levels(trace, level_set, pair):
    _lib, L, dl = _L()
    shapes, a, B = LEVEL_SETS[level_set], 3, 2
    rs = np.random.RandomState(len(shapes) * 10 + LEVEL_PAIRS.index(pair))
    lg, bb, top, A = _level_tensors(rs, B, shapes, a)
    ldt, bdt = (BF16 if t == "bf16" else F32 for t in pair.split("+"))
    if ldt == BF16:
        lg = [bf16_round(t) for t in lg]
    if bdt == BF16:
        bb = [bf16_round(t) for t in bb]
    anchors = _synth.rois_log_uniform(rs, B, A, lo=8, hi=200).astype(f32)
    pre, post = max(len(top), A // 2), 40
    K = min(pre, A)
    tl, tbb, ta = [cu(t).to(ldt) for t in lg], [cu(t).to(bdt) for t in bb], cu(anchors)
    out = sent_f32((B, post, 4))
    d, dbg = _prop_debug(dl, B, K, post)
    params = _prop_params(pre, post)
    n = len(shapes)
    pl, pb = (ctypes.c_void_p * n)(*[dl(t) for t in tl]), (ctypes.c_void_p * n)(*[dl(t) for t in tbb])

    def call():
        ws = poison(L.od_proposal_levels_workspace_bytes(B, A, ctypes.byref(params)), ta.device)
        _lib.check(L.od_proposal_forward_levels(pl, pb, n, dl(ta), None, ctypes.byref(params), dl(out), ctypes.byref(dbg),
                                                ws.data_ptr(), ws.numel(), _lib.stream_ptr(ta.device)),
                   "od_proposal_forward_levels")
    _, names = trace(call)
    probs, flat = oracle.rpn_levels_to_flat(lg, bb)
    want, wd = oracle.proposal_forward(probs, flat, anchors, STD, pre, post, 0.7, debug=True)
    _check_prop(out, d, want, wd, K)
    assert (np.sort(wd["ix"][:, :len(top)], 1) == np.array(top)).all(), "the edge anchors must be the top scores"
    return names


# ------------------------------------------------------------------ roi_pool
def run_roi_pool(trace, n, D):
    _lib, L, dl = _L()
    rs = np.random.RandomState(n * 7 + D)
    B, h, w, image_h, image_w = 2, 38, 63, 600.0, 1000.0
    fmap = rs.random_sample((B, h, w, D)).astype(f32)
    xy1 = rs.uniform(-20, 900, (n, 2))
    wh = rs.uniform(0, 300, (n, 2))
    rois = np.concatenate([rs.randint(0, B, (n, 1)), xy1, xy1 + wh], 1).astype(f32)
    border = np.array([[0, 0, 0, 999, 599], [1, 0, 0, 0, 0], [1, 999, 599, 999, 599], [0, 990, 0, 1200, 700],
                       [1, -30, 580, 40, 620]], f32)                            # whole image, corners, past the edges
    m = min(len(border), n)
    rois[n - m:] = border[:m]
    rois[n - 1, 0] = B - 1                                                     # the last row on the last image
    bad = np.zeros(n, bool)
    if n >= 3:
        rois[n - 3, 0] = B                                                     # out of range: zeros
        bad[n - 3] = True
    tf, tr = cu(fmap), cu(rois)
    out = sent_f32((n, 7, 7, D))

    def call():
        _lib.check(L.od_roi_pool_forward(dl(tf), dl(tr), image_h, image_w, dl(out), _lib.stream_ptr(tf.device)),
                   "od_roi_pool_forward")
    _, names = trace(call)
    got = host(out)
    assert_bits(got, oracle.roi_pool(fmap, rois, image_h, image_w), f"roi_pool n={n} D={D}")
    assert_written(got, "pooled")
    assert not got[bad].any()
    boxes = np.stack([rois[:, 2] / image_h, rois[:, 1] / image_w, rois[:, 4] / image_h, rois[:, 3] / image_w], 1)
    bi = rois[:, 0].astype(np.int32)
    bi[bad] = 0
    crops, ok = crop_and_resize_f64(fmap, boxes, bi, 14, 14)
    want = crops.reshape(n, 7, 2, 7, 2, D).max(axis=(2, 4))
    ok = ok.reshape(n, 7, 2, 7, 2).all(axis=(2, 4)) & ~bad[:, None, None]
    if ok.any():
        err = np.abs(got.astype(f64) - want)[ok]
        assert err.max() <= 1e-4, f"roi_pool n={n} D={D}: max |cuda - fp64| = {err.max():.3e}"
    return names


# ------------------------------------------------------------------ bf16 ROIAlign
def run_crop_dt(trace, n, crop, D, pair):
    """od_crop_and_resize on bf16 maps and / or a bf16 output against the oracle and the fp32 call on the widened maps;
    crops with an out-of-range box_ind stay untouched."""
    _lib, L, dl = _L()
    md, od = BY_PAIR_ID[pair]
    rs = np.random.RandomState(n * 13 + D + crop[0])
    img = bf16_round(rs.random_sample((3, 19, 23, D)))
    boxes = _synth.random_boxes(rs, n, flip=True)
    hard = np.array([[0, 0, 1, 1], [0.3, 0.3, 0.3, 0.3], [-0.2, -0.1, 0.5, 0.5], [0.5, 0.5, 1.3, 1.2],
                     [0.9, 0.8, 0.1, 0.2], [0, 0, 0, 0]], f32)
    m = min(len(hard), n)
    boxes[n - m:] = hard[:m]
    bi = rs.randint(0, 3, n).astype(np.int32)
    skip = np.zeros(n, bool)
    if n >= 3:
        bi[n - 2], bi[0] = 3, -1
        skip[[0, n - 2]] = True
    tbx, tbi = cu(boxes), cu(bi)

    def call(mdt, odt):
        ti = cu(img).to(mdt)
        out = sent_out((n, crop[0], crop[1], D), odt)
        _, names = trace(lambda: _lib.check(L.od_crop_and_resize(dl(ti), dl(tbx), dl(tbi), crop[0], crop[1], 0.5, dl(out),
                                                                 _lib.stream_ptr(ti.device)), "od_crop_and_resize"))
        return out, names
    want = oracle.crop_and_resize(img, boxes, bi, crop[0], crop[1], extrapolation=0.5)
    ref, _ = call(F32, F32)
    ref = check_out(ref, want, F32, "fp32 call", skip)
    out, names = call(md, od)
    check_out(out, want, od, f"{pair} vs oracle", skip)
    check_out(out, ref, od, f"{pair} vs fp32 call", skip)
    return names


def run_pyramid_dt(trace, N, pair):
    """od_pyramid_roi_align_forward_ws (B = 1, 14x14, D = 256) on a bf16 dtype pair; n >= 512 also through _ordered
    with the order od_roi_processing_order gives."""
    _lib, L, dl = _L()
    md, od = BY_PAIR_ID[pair]
    rs = np.random.RandomState(N + 5)
    fmaps = [bf16_round(f) for f in _roi_maps(rs, 1)]
    props = _edge_rois(rs, 1, N)
    pr = cu(props)
    dev = pr.device
    want, wlv = oracle.pyramid_roi_align(fmaps, props, 1024, 1024, 14, 14)
    want = want[0]
    order_ws = N > 100                                                         # the mask branch has no order workspace
    zws = _lib.zeroed_workspace(L.od_pyramid_roi_align_workspace_bytes_n(N) if order_ws else
                                L.od_pyramid_roi_align_workspace_bytes(), dev)
    assert int(zws[:256].count_nonzero()) == 0

    def call(mdt, odt, order=None):
        fm = [cu(f).to(mdt) for f in fmaps]
        ptrs = (ctypes.c_void_p * 4)(*[dl(f) for f in fm])
        out, lv = sent_out((1, N, 14, 14, 256), odt), sent_i32((1, N))

        def go():
            zws[256:].fill_(0xFF)
            if order is None:
                rc = L.od_pyramid_roi_align_forward_ws(ptrs, 4, 2, dl(pr), 1024, 1024, 14, 14, dl(out), dl(lv),
                                                       zws.data_ptr(), zws.numel(), _lib.stream_ptr(dev))
            else:
                rc = L.od_pyramid_roi_align_forward_ordered(ptrs, 4, 2, dl(pr), 1024, 1024, 14, 14, dl(out), dl(lv),
                                                            dl(order), zws.data_ptr(), zws.numel(), _lib.stream_ptr(dev))
            _lib.check(rc, "od_pyramid_roi_align_forward_ws / _ordered")
        _, names = trace(go)
        assert int(zws[:256].count_nonzero()) == 0, "the ticket bytes were not left zeroed"
        assert np.array_equal(host(lv), wlv)
        return out[0], names
    ref, _ = call(F32, F32)
    ref = check_out(ref, want, F32, "fp32 call")
    out, names = call(md, od)
    check_out(out, want, od, f"{pair} vs oracle")
    check_out(out, ref, od, f"{pair} vs fp32 call")
    if N >= 512:
        order = sent_i32((N,))
        _lib.check(L.od_roi_processing_order(dl(pr), 1024, 1024, 2, 4, dl(order), _lib.stream_ptr(dev)),
                   "od_roi_processing_order")
        assert np.array_equal(np.sort(host(order)), np.arange(N))
        out2, names2 = call(md, od, order)
        check_out(out2, want, od, f"{pair} _ordered vs oracle")
        assert_launched(names2, must=[f"od::crop_rows_kernel<{TNAME[md]},{TNAME[od]}>("], must_not=["od::roi_order_kernel("])
    return names


# ------------------------------------------------------------------ bf16 heads
def head_case(trace, name, v):
    pair = BY_HEAD_PAIR_ID[v[0]]
    if name == "bf16_det":
        row, val = v[1], v[2]
        names, _ = (run_detection(trace, 2048, kept=val, dts=pair) if row == "det_finalize_kept" else
                    run_detection(trace, val, dts=pair))
        return names
    run = run_rpn_loss if name == "bf16_rpn_loss" else run_mrcnn_loss
    names, got = run(trace, v[1], dts=pair)
    _, ref = run(trace, v[1], dts=(F32, F32), vals=pair)                        # the fp32 call on the widened inputs
    for i, (g, r) in enumerate(zip(got, ref)):
        assert np.array_equal(np.ascontiguousarray(g).view(np.uint32), np.ascontiguousarray(r).view(np.uint32)), \
            f"output {i} differs from the fp32 call"
    return names


# ------------------------------------------------------------------ the GPU cases
@pytest.mark.gpu
@pytest.mark.parametrize("name,value", CASES)
def test_front_boundary(_cuda, kernel_trace, name, value):
    b = BY_NAME[name]
    v = tuple(resolve(x) if str(x).startswith("sms") else x for x in value) if isinstance(value, tuple) else resolve(value)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    if name.startswith("frcnn_"):
        names = frcnn_case(kernel_trace, name, v)
    elif name == "proposal_k_vs_a":
        names, _ = run_proposals(kernel_trace, v[0], 2, A_PROP, v[1], 300)
    elif name == "proposal_n_vs_k":
        names, wd = run_proposals(kernel_trace, v[0], 2, A_PROP, K_PROP, v[1])
        assert (wd["num_kept"] > K_PROP // 2).all()
    elif name == "proposal_grids":
        names, _ = run_proposals(kernel_trace, v[0], 1, 600, v[1], v[1])
    elif name == "levels_edges":
        names = run_levels(kernel_trace, *v)
    elif name == "roi_pool_bins":
        names = run_roi_pool(kernel_trace, *v)
    elif name == "bf16_crop_rows_grid":
        names = run_crop_dt(kernel_trace, v[1], (14, 14), 256, v[0])
    elif name in ("bf16_mask_branch", "bf16_roi_order"):
        names = run_pyramid_dt(kernel_trace, v[1], v[0])
    elif name == "bf16_tier":
        names = run_crop_dt(kernel_trace, 40, (1, 1), v[1], v[0])
    elif name == "bf16_bins_32":
        names = run_crop_dt(kernel_trace, v[1], (1, 1), 128, v[0])
    elif name == "bf16_bins_512":
        names = run_crop_dt(kernel_trace, v[1], (1, 1), 8, v[0])
    elif name in ("bf16_det", "bf16_rpn_loss", "bf16_mrcnn_loss"):
        names = head_case(kernel_trace, name, v)
    else:
        raise AssertionError(f"no runner for {name}")
    if b.kernels is not None:
        must, must_not = b.kernels(v, sms)
        assert_launched(names, must=must, must_not=must_not)
