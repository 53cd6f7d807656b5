"""Size boundaries: every place where host code changes its launch plan, or where a kernel's tile, chunk or CTA ends, run
on both sides, through the C ABI, against the CPU oracle.

BOUNDARIES holds one row per boundary: the entry point, the size parameter, the values on each side, the source constant
or expression they come from and, for a dispatch threshold, the kernels expected on each side. The values are computed
here from Python restatements of the host planning code (NMS ring slots and the staged / unstaged / wide choice, the
two-round rule, top-k's cand_capacity / blocks_per_row / index_bits, the ROIAlign tier and crop_rows_serves) over the
constants in CONST. test_boundary_constants_match_sources (no GPU) reads those constants and the literal thresholds from
objectdetection_b200/csrc and fails when one of them changes and the table does not follow.

Two numbers of SMs appear. The crop_rows_kernel grid (min(n_rois, SMs)) and the slice of the cooperative wide NMS scan are
planned on the device's multiprocessor count at run time: those rows name their values as "sms-1", "sms", "sms+1" and
resolve them on the GPU. top-k's blocks_per_row uses the compiled constant kNumSMsB200 (CONST), so its edge is fixed.

Every GPU case owns its output tensors and pre-fills them with a sentinel bit pattern (float 0x7FBADBAD, int32 0x7EADBEEF),
fills the stream's cached workspace with 0xFF bytes before the call (for ROIAlign: everything after the 256 ticket bytes,
which must stay zero and are checked to be zero again afterwards), compares every main output with the oracle bit for bit,
padding included, and checks from the raw bits that no sentinel word survives outside the documented untouched regions
(crops with an out-of-range box_ind). Each dispatch threshold reads the kernel trace on both sides."""
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
from objectdetection_b200.config import config as Conf  # noqa: E402
from test_gpu_dispatch import _assert_close_f64, _cuda, assert_launched, kernel_trace  # noqa: E402,F401
from test_gpu_parity import assert_bits, cu, host  # noqa: E402

torch = pytest.importorskip("torch")
f32 = np.float32
F32, BF16 = torch.float32, torch.bfloat16
CSRC = os.path.join(os.path.dirname(HERE), "objectdetection_b200", "csrc")

F_SENT, I_SENT = 0x7FBADBAD, 0x7EADBEEF

# ------------------------------------------------------------------ constants of the planning code
# name -> (file, value). Parsed from `constexpr <type> name = <expr>;` by test_boundary_constants_match_sources.
CONST = {
    "kTileKeys": ("topk.cu", 1024),
    "kMergeMaxK": ("topk.cu", 16384),
    "kSmemSortMax": ("topk.cu", 16384),
    "kNumSMsB200": ("common.cuh", 148),
    "kIouThreads": ("targets.cu", 256),
    "kTgtThreads": ("targets.cu", 1024),
    "kDetRankMine": ("detection.cu", 64),
    "kDetRankTile": ("detection.cu", 1024),
    "kFinThreads": ("detection.cu", 1024),
    "kLossChunk": ("losses.cu", 1024),
    "kChunk": ("rpn_targets.cu", 1024),
    "kFusedMaxGt": ("rpn_targets.cu", 256),
    "kBinBins": ("roi_align.cu", 32),
    "kRowsMinPool": ("roi_align.cu", 10),
    "kRowsMaxPool": ("roi_align.cu", 16),
    "kRowsMaxWidth": ("roi_align.cu", 14),
    "kRowsD4": ("roi_align.cu", 64),
    "kOrderThreads": ("roi_align.cu", 1024),
    "kOrderPerThread": ("roi_align.cu", 4),
    "kScanMaxSlots": ("nms.cu", 8),
    "kWidePrefetchMaxS": ("nms.cu", 16),
}
# literal thresholds the formulas below restate, as they stand in the sources (whitespace-insensitive)
LITERALS = [
    ("nms.cu", "const size_t kSmemBudget = 200 * 1024;"),                 # the staged scan's shared-memory budget
    ("nms.cu", "if (W <= 32 && nslots > 4) nslots = 4;"),                 # short rows: four slots
    ("nms.cu", "plain + 2 * per_slot <= kSmemBudget"),                    # staged needs two slots
    ("nms.cu", "const bool two_rounds = c1 + 8 <= W;"),                   # the two-round rule
    ("nms.cu", "int c1 = (int)((max_out + max_out / 2 + 63) / 64);"),
    ("nms.cu", "return wide_scan_smem(S, 2) <= 200 * 1024 ? 2 : 1;"),
    ("nms.cu", "int64_t G = (W + 3) / 4;"),                               # wide scan: at least four words per CTA
    ("nms.cuh", "return (((K + 63) / 64) + 1) & ~(int64_t)1;"),           # mask stride
    ("topk.cu", "const int64_t by_work = (cols + 2047) / 2048;"),
    ("topk.cu", "const int64_t by_fill = (2 * kNumSMsB200 + rows - 1) / rows;"),
    ("topk.cu", "int64_t cap = 4 * next_pow2(k > 0 ? k : 1);"),
    ("topk.cu", "if (cap < 16384) cap = 16384;"),
    ("topk.cu", "const bool overflow = n_cand > (uint32_t)cand_cap;"),
    ("topk.cuh", "while (((int64_t)1 << ib) < cols) ++ib;"),
    ("roi_align.cu", "n_rois >= 512 && src.rois_per_image <= kOrderThreads * kOrderPerThread"),
    ("roi_align.cu", "n_rois < (int64_t)sms[dev] ? n_rois : (int64_t)sms[dev]"),
    ("roi_align.cu", "if (lg >= 0 && D4 >= 16) {"),
    ("roi_align.cu", "constexpr int BINS = 512;"),
    ("targets.cu", "if (smem_iou + iou_static > 48 * 1024)"),           # static + dynamic shared memory past 48 KiB
    ("targets.cu", "constexpr int kIouRows = kIouThreads / 4;"),
    ("detection.cu", "if (N <= 4096) {"),
    ("topk.cu", "if (smem + merge_static > 48 * 1024)"),
]


# static shared memory (bytes) of the kernels whose dynamic opt-in edge depends on it, as ptxas lays them out for sm_100a;
# a launch without the opt-in gets 48 KiB, static and dynamic together
STATIC_SMEM = {"detection_iou_kernel": 1456, "topk_merge_emit_kernel": 1024}


def C(name):
    return CONST[name][1]


# ------------------------------------------------------------------ the planning formulas, restated
def nms_slots(K):
    """scan_round_launch: ring slots of the staged scan (0 = not staged)."""
    W = (K + 63) // 64
    Ws = (W + 1) & ~1
    plain, per_slot, budget = ((W + 15) & ~15) * 8, (64 * Ws + 64) * 8, 200 * 1024
    if plain + 2 * per_slot > budget:
        return 0
    n = min(C("kScanMaxSlots"), (budget - plain) // per_slot)
    return 4 if W <= 32 and n > 4 else n


def nms_two_rounds(K, max_out):
    return (max_out + max_out // 2 + 63) // 64 + 8 <= (K + 63) // 64


def nms_scan_kernel(B, K, max_out, sms):
    """The scan kernel one od_nms call launches (runtime SM count for the wide scan's slice)."""
    if nms_slots(K) >= 2:
        return "od::nms_scan_kernel<true>("
    W = (K + 63) // 64
    if nms_two_rounds(K, max_out) or W < 64:
        return "od::nms_scan_kernel<false>("
    G = min((W + 3) // 4, sms // B)
    S = (W + G - 1) // G
    return "od::nms_scan_wide_kernel<true>(" if S <= C("kWidePrefetchMaxS") else "od::nms_scan_wide_kernel<false>("


def slot_edges(lo=1, hi=20000):
    """Every K where the ring slot count changes while the scan stays staged."""
    return [K for K in range(lo + 1, hi) if nms_slots(K) != nms_slots(K - 1) and nms_slots(K)]


def index_bits(cols):
    ib = 1
    while (1 << ib) < cols:
        ib += 1
    return ib


def next_pow2(v):
    p = 1
    while p < v:
        p <<= 1
    return p


def cand_capacity(cols, k):
    return min(max(4 * next_pow2(max(k, 1)), 16384), cols)


def blocks_per_row(rows, cols):
    return max(1, min((cols + 2047) // 2048, (2 * C("kNumSMsB200") + rows - 1) // rows))


def crop_rows_serves(ph, pw, D):
    return (D == 4 * C("kRowsD4") and ph <= C("kRowsMaxPool") and pw <= C("kRowsMaxWidth")
            and max(ph, pw) >= C("kRowsMinPool"))


def roi_order_runs(n_rois, rois_per_image):
    return n_rois >= 512 and rois_per_image <= C("kOrderThreads") * C("kOrderPerThread")


def bins_tier(D):
    """fp32 maps: the crop_bins CTA size (bins) for depth D."""
    D4 = D // 4
    return C("kBinBins") if D4 & (D4 - 1) == 0 and D4 >= 16 else 512


def gt_smem_opt_in(G):
    return G * 16 + STATIC_SMEM["detection_iou_kernel"] > 48 * 1024


IOU_EDGE = next(G for G in range(1, 8193) if gt_smem_opt_in(G))
MERGE_EDGE = next(k for k in range(1, C("kMergeMaxK")) if 8 * k + STATIC_SMEM["topk_merge_emit_kernel"] > 48 * 1024)


def sides(edge, lo=1, hi=0):
    """Values around an edge: edge - lo .. edge + hi."""
    return list(range(edge - lo, edge + hi + 1))


# ------------------------------------------------------------------ the table
class Boundary:
    def __init__(self, name, entry, param, values, source, kernels=None):
        self.name, self.entry, self.param, self.values, self.source = name, entry, param, values, source
        self.kernels = kernels          # (value, runtime SMs) -> (must, must_not), or None where the kernels do not change


NMS_SLOT_EDGES = slot_edges()
NMS_STAGED_LIMIT = next(K for K in range(1, 40000) if nms_slots(K) == 0)
_two = next(m for m in range(6000, 0, -1) if nms_two_rounds(6000, m))
TOPK_CAP = cand_capacity(40000, 1000)

BOUNDARIES = [
    Boundary("nms_ring_slots", "od_nms", "K (max_out = K)", [v for e in NMS_SLOT_EDGES for v in (e - 1, e)],
             "scan_round_launch: nslots = min(kScanMaxSlots, (200 KiB - plain) / per_slot), 4 when W <= 32",
             kernels=lambda v, sms: (["od::nms_scan_kernel<true>("], ["od::nms_scan_wide_kernel<", "od::nms_scan_kernel<false>("])),
    Boundary("nms_staged_limit", "od_nms", "K (max_out = K)", [NMS_STAGED_LIMIT - 1, NMS_STAGED_LIMIT],
             "scan_round_launch: plain + 2 * per_slot <= 200 KiB; past it the cooperative wide scan (runtime SM count)",
             kernels=lambda v, sms: ([nms_scan_kernel(2, v, v, sms)],
                                     ["od::nms_scan_kernel<false>("] + (["od::nms_scan_wide_kernel<"] if nms_slots(v) else
                                                                        ["od::nms_scan_kernel<true>("]))),
    Boundary("nms_two_rounds", "od_nms", "max_out (K = 6000)", [_two, _two + 1],
             "nms_sorted_launch: two rounds iff ceil(1.5 max_out / 64) + 8 <= W",
             kernels=lambda v, sms: (["od::nms_scan_kernel<true>("], ["od::nms_scan_wide_kernel<"])),
    Boundary("topk_merge_smem", "od_topk", "k (cols = 8000)", [MERGE_EDGE - 1, MERGE_EDGE, 6144, 6145],
             "topk_launch: k * 8 bytes of merge keys plus the kernel's static shared memory opt in past 48 KiB"),
    Boundary("topk_tile", "od_topk", "k (cols = 5000)", sides(C("kTileKeys"), 1, 1) + sides(2 * C("kTileKeys"), 1, 1),
             "topk_tile_sort_kernel: kTileKeys keys per tile; the merge takes ceil(k / kTileKeys) tiles"),
    Boundary("topk_merge_max", "od_topk", "k (cols = 20000)", [C("kMergeMaxK"), C("kMergeMaxK") + 1],
             "topk_launch: k <= kMergeMaxK tile sort + merge, else the global bitonic sort",
             kernels=lambda v, sms: ((["od::topk_tile_sort_kernel(", "od::topk_merge_emit_kernel("],
                                      ["od::bitonic_step_global_kernel(", "od::pad_emit_kernel("]) if v <= C("kMergeMaxK") else
                                     (["od::bitonic_step_global_kernel(", "od::pad_emit_kernel("],
                                      ["od::topk_tile_sort_kernel(", "od::topk_merge_emit_kernel("]))),
    Boundary("topk_index_bits", "od_topk", "cols (k = 1000)", [4095, 4096, 4097, 65535, 65536, 65537],
             "index_bits(cols): the key's index field widens past each power of two"),
    Boundary("topk_cand_capacity", "od_topk", "keys in the threshold bucket (cols = 40000, k = 1000)",
             [TOPK_CAP, TOPK_CAP + 1], "cand_capacity(cols, k) = min(max(4 next_pow2(k), 16384), cols); overflow iff n_cand > cap"),
    Boundary("topk_blocks_cols", "od_topk", "cols (rows = 2, k = 1000)", [2048, 2049],
             "blocks_per_row: by_work = ceil(cols / 2048)"),
    Boundary("topk_blocks_rows", "od_topk", "rows (cols = 5000, k = 1000)", [2 * C("kNumSMsB200") - 1, 2 * C("kNumSMsB200")],
             "blocks_per_row: by_fill = ceil(2 kNumSMsB200 / rows) (compiled constant, not the runtime count)"),
    Boundary("crop_rows_grid", "od_crop_and_resize", "n_rois (14x14, D = 256)", [1, "sms-1", "sms", "sms+1"],
             "launch_crop_rows: grid = min(n_rois, runtime SMs)",
             kernels=lambda v, sms: (["od::crop_rows_kernel("], ["od::crop_bins_kernel<"])),
    Boundary("roi_align_mask_branch", "od_pyramid_roi_align_forward_ws", "B*N (B = 1, 14x14, D = 256, ticket workspace)",
             [1, 100, "sms-1", "sms", "sms+1"], "the mask branch pools <= 100 detections of an image; grid = min(n_rois, SMs)",
             kernels=lambda v, sms: (["od::crop_rows_kernel("], ["od::roi_order_kernel(", "od::crop_bins_kernel<"])),
    Boundary("roi_order_n", "od_pyramid_roi_align_forward_ws", "n_rois (B = 1, 14x14, D = 256)", [511, 512],
             "launch_crop_bins: the order pre-pass needs n_rois >= 512",
             kernels=lambda v, sms: ((["od::roi_order_kernel(", "od::crop_rows_kernel("], []) if roi_order_runs(v, v) else
                                     (["od::crop_rows_kernel("], ["od::roi_order_kernel("]))),
    Boundary("roi_order_per_image", "od_pyramid_roi_align_forward_ws", "rois_per_image (B = 1, 7x7, D = 256)",
             [C("kOrderThreads") * C("kOrderPerThread"), C("kOrderThreads") * C("kOrderPerThread") + 1],
             "launch_crop_bins: rois_per_image <= kOrderThreads * kOrderPerThread",
             kernels=lambda v, sms: ((["od::roi_order_kernel(", "od::crop_bins_kernel<32, 2, true, true>("],
                                      ["od::crop_bins_kernel<32, 2, true, false>("]) if roi_order_runs(v, v) else
                                     (["od::crop_bins_kernel<32, 2, true, false>("],
                                      ["od::roi_order_kernel(", "od::crop_bins_kernel<32, 2, true, true>("]))),
    Boundary("crop_bins_32", "od_crop_and_resize", "total_bins (1x1 crops, D = 64)",
             [2 * C("kBinBins") - 1, 2 * C("kBinBins"), 2 * C("kBinBins") + 1],
             "crop_bins_kernel<kBinBins = 32>: the last CTA's bins",
             kernels=lambda v, sms: (["od::crop_bins_kernel<32, 2, true, false>("], ["od::crop_bins_kernel<512,"])),
    Boundary("crop_bins_512", "od_crop_and_resize", "total_bins (1x1 crops, D = 8)", [511, 512, 513],
             "crop_bins_kernel<BINS = 512> (thin depth): the last CTA's bins",
             kernels=lambda v, sms: (["od::crop_bins_kernel<512, 2, true, false>("], ["od::crop_bins_kernel<32,"])),
    Boundary("targets_gt_smem", "od_detection_target_forward", "G (N = 300)", [IOU_EDGE - 1, IOU_EDGE, 3072, 3073],
             "detection_iou_kernel: G * 16 bytes of GT table plus the kernel's static shared memory opt in past 48 KiB"),
    Boundary("targets_iou_rows", "od_detection_target_forward", "N (G = 20)", sides(C("kIouThreads") // 4, 1, 1),
             "detection_iou_kernel: kIouRows = kIouThreads / 4 proposals per CTA"),
    Boundary("targets_compaction", "od_detection_target_forward", "N (G = 20)", sides(C("kTgtThreads"), 1, 1),
             "detection_target_kernel: one kTgtThreads CTA compacts the N proposals"),
    Boundary("targets_rois", "od_detection_target_forward", "R (N = 3200, G = 60)", [C("kTgtThreads"), C("kTgtThreads") + 1],
             "detection_target_kernel: one kTgtThreads CTA writes the R rows"),
    Boundary("det_rank_tile", "od_detection_forward", "N", [C("kDetRankTile"), C("kDetRankTile") + 1],
             "det_rank_gather_kernel: kDetRankTile keys per rank tile",
             kernels=lambda v, sms: (["od::det_rank_gather_kernel("], ["od::det_gather_kernel("])),
    Boundary("det_rank_vs_sort", "od_detection_forward", "N", [4096, 4097],
             "od_detection_forward: N <= 4096 rank gather, else bitonic sort + gather",
             kernels=lambda v, sms: ((["od::det_rank_gather_kernel("], ["od::det_gather_kernel(", "od::sort_u64_smem_kernel("])
                                     if v <= 4096 else
                                     (["od::sort_u64_smem_kernel(", "od::det_gather_kernel("], ["od::det_rank_gather_kernel("]))),
    Boundary("det_scan_short_rows", "od_detection_forward", "N", [2048, 2049],
             "scan_round_launch: W <= 32 caps the ring at 4 slots"),
    Boundary("det_finalize_kept", "od_detection_forward", "rows kept before NMS (N = 2048)", sides(C("kFinThreads"), 1, 1),
             "det_finalize_kernel: kFinThreads positions per prefix / compaction tile"),
    Boundary("rpn_loss_chunk", "od_rpn_loss_forward", "A (B = 2)", sides(C("kLossChunk"), 1, 1) + sides(2 * C("kLossChunk"), 1, 1),
             "rpn_loss_class_kernel / rpn_loss_box_kernel: kLossChunk anchors per CTA"),
    Boundary("mrcnn_loss_cta", "od_mrcnn_loss_forward", "B*R (B = 1)", sides(1024, 1, 1),
             "mrcnn_loss_kernel: one 1024-thread CTA loops over B*R"),
    Boundary("rpn_target_chunk", "od_rpn_target_forward", "A (G = 12)", sides(C("kChunk"), 1, 1),
             "rpn_count / compact / perm kernels: kChunk anchors per CTA"),
    Boundary("rpn_target_fused_gt", "od_rpn_target_forward", "G (A = 3000)", [C("kFusedMaxGt"), C("kFusedMaxGt") + 1],
             "od_rpn_target_forward: G <= kFusedMaxGt fuses the per-GT arg-max into the anchor pass",
             kernels=lambda v, sms: ((["od::rpn_anchor_best_kernel<true>(", "od::rpn_gt_reduce_kernel("],
                                      ["od::rpn_anchor_best_kernel<false>(", "od::rpn_gt_best_kernel("]) if v <= C("kFusedMaxGt") else
                                     (["od::rpn_anchor_best_kernel<false>(", "od::rpn_gt_best_kernel("],
                                      ["od::rpn_anchor_best_kernel<true>(", "od::rpn_gt_reduce_kernel("]))),
]
BY_NAME = {b.name: b for b in BOUNDARIES}
CASES = [pytest.param(b.name, v, id=f"{b.name}-{v}") for b in BOUNDARIES for v in b.values]


# ------------------------------------------------------------------ no GPU: the table follows the sources
def _flat(s):
    return re.sub(r"\s+", "", s)


def parse_constants(consts=CONST, csrc=CSRC):
    """Values of the `consts` names as the sources define them (simple constexpr expressions over earlier constants)."""
    got = {}
    for name, (fname, _) in consts.items():
        src = open(os.path.join(csrc, fname)).read()
        m = re.search(rf"constexpr\s+[\w:]+\s+{name}\s*=\s*([^;]+);", src)
        assert m, f"{name} is not defined in {fname}"
        expr = m.group(1)
        env = {k: v for k, v in got.items()}
        for dep in re.findall(r"\bk\w+", expr):
            if dep not in env:
                dm = re.search(rf"constexpr\s+[\w:]+\s+{dep}\s*=\s*([^;]+);", src)
                assert dm, f"{name}: {dep} not found in {fname}"
                env[dep] = eval(dm.group(1), {}, env)
        got[name] = eval(expr, {}, env)
    return got


def check_sources(consts, literals, csrc=CSRC):
    """Every (file, value) of `consts` is what the sources define, and every (file, text) of `literals` is still in its
    file (whitespace-insensitive): a table built on them restates the planning code as it stands."""
    parsed = parse_constants(consts, csrc)
    wrong = {n: (parsed[n], v) for n, (_, v) in consts.items() if parsed[n] != v}
    assert not wrong, f"constants changed in the sources (now, table): {wrong}; update the constants and the formulas"
    missing = [(f, s) for f, s in literals if _flat(s) not in _flat(open(os.path.join(csrc, f)).read())]
    assert not missing, f"thresholds the table restates are no longer in the sources: {missing}"


def test_boundary_constants_match_sources():
    check_sources(CONST, LITERALS)


def test_boundary_table_values():
    """The computed values are the edges the planning code has: each boundary has a value on each side, and the
    restated formulas change exactly there."""
    assert NMS_SLOT_EDGES == [2049, 3073, 3585, 4097, 4993, 6273, 8321], NMS_SLOT_EDGES
    assert NMS_STAGED_LIMIT == 12545
    assert nms_slots(12544) == 2 and nms_slots(2048) == 4 and nms_slots(2049) == 8
    assert _two == 3669 and nms_two_rounds(6000, 3669) and not nms_two_rounds(6000, 3670)
    assert nms_scan_kernel(2, 12545, 12545, 148) == "od::nms_scan_wide_kernel<true>("
    assert [index_bits(c) for c in (4095, 4096, 4097, 65535, 65536, 65537)] == [12, 12, 13, 16, 16, 17]
    assert TOPK_CAP == 16384
    assert blocks_per_row(2, 2048) == 1 and blocks_per_row(2, 2049) == 2
    assert blocks_per_row(295, 5000) == 2 and blocks_per_row(296, 5000) == 1
    assert crop_rows_serves(14, 14, 256) and not crop_rows_serves(7, 7, 256)
    assert not roi_order_runs(511, 511) and roi_order_runs(512, 512) and not roi_order_runs(4097, 4097)
    assert bins_tier(64) == 32 and bins_tier(8) == 512
    assert IOU_EDGE == 2982 and gt_smem_opt_in(3072) and MERGE_EDGE == 6017
    for b in BOUNDARIES:
        assert len(b.values) >= 2 and len(set(map(str, b.values))) == len(b.values), b.name
        assert b.source and b.entry.startswith("od_"), b.name


# ------------------------------------------------------------------ GPU helpers
def sent_f32(shape):
    return torch.full(shape, F_SENT, dtype=torch.int32, device="cuda").view(torch.float32)


def sent_i32(shape):
    return torch.full(shape, I_SENT, dtype=torch.int32, device="cuda")


def sent_f64(shape):
    return torch.full(shape, (F_SENT << 32) | F_SENT, dtype=torch.int64, device="cuda").view(torch.float64)


def assert_written(a, what, untouched=None):
    """No sentinel word outside `untouched` (a boolean mask over the leading axes); every word inside it untouched."""
    a = np.ascontiguousarray(a)
    words = a.view(np.uint32).reshape(a.shape[:1] + (-1,)) if a.dtype.itemsize >= 4 else None
    sent = F_SENT if a.dtype != np.int32 else I_SENT
    hit = words == sent
    if untouched is None:
        untouched = np.zeros(a.shape[0], bool)
    bad = np.argwhere(hit & ~untouched.reshape(-1, 1))
    assert bad.size == 0, f"{what}: {bad.shape[0]} words still hold the sentinel, first at {bad[:3].tolist()}"
    assert hit[untouched].all(), f"{what}: rows that must stay untouched were written"


def bf16_round(a):
    """The bf16 value nearest to each element (round to nearest even, as torch converts), as fp32."""
    return torch.from_numpy(np.ascontiguousarray(a, f32)).to(BF16).float().numpy()


def head_inputs(arrays, dts, vals):
    """Head-output arrays for a call on dtypes `dts`: each array whose entry in `vals` is BF16 holds bf16 values (so that
    the fp32 reference sees the widened inputs); returns (host arrays, CUDA tensors of dtypes dts)."""
    arrays = [bf16_round(a) if v == BF16 else a for a, v in zip(arrays, vals)]
    return arrays, [cu(a).to(dt) for a, dt in zip(arrays, dts)]


def poison(nbytes, dev):
    from objectdetection_b200 import _lib
    ws = _lib.workspace(nbytes, dev)
    ws.fill_(0xFF)
    return ws


def resolve(v):
    if isinstance(v, str):
        sms = torch.cuda.get_device_properties(0).multi_processor_count
        return sms + int(v[3:] or 0)
    return v


def _L():
    from objectdetection_b200 import _lib
    return _lib, _lib.lib(), _lib.DL()


# ------------------------------------------------------------------ runners, one per entry point
def _nms_inputs(rs, B, K):
    """Image 0 clustered (few survivors), image 1 sparse (many); hard rows in the last, partial 64-box chunk:
    duplicates, zero area, flipped, tied scores; ragged num_valid."""
    from test_gpu_dispatch import _clustered_boxes
    boxes = np.stack([_clustered_boxes(rs, K), _synth.rois_log_uniform(rs, 1, K, image=4096, lo=4, hi=48)[0]][:B])
    scores = (rs.randint(0, 4000, (B, K)) / 4000).astype(f32)
    t = K - 1 - (K - 1) % 64                                    # first box of the last chunk
    for b in range(B):
        last = np.arange(t, K)
        boxes[b, last[::3]] = boxes[b, last[0]]                  # duplicates
        boxes[b, K - 1, 2:] = boxes[b, K - 1, :2]                # zero area
        if K - t > 2:
            boxes[b, K - 2] = boxes[b, K - 2][[2, 3, 0, 1]]      # flipped
        scores[b, last[1::2]] = scores[b, t]                     # ties
    nv = np.array([K, K - 37 if K > 100 else K], np.int32)[:B]
    return boxes, scores, nv


def run_nms(trace, K, max_out):
    _lib, L, dl = _L()
    rs = np.random.RandomState(K * 7 + max_out)
    B = 2
    boxes, scores, nv = _nms_inputs(rs, B, K)
    tb, ts, tn = cu(boxes), cu(scores), cu(nv)
    keep, num = sent_i32((B, max_out)), sent_i32((B,))

    def call():
        ws = poison(L.od_nms_workspace_bytes(B, K), tb.device)
        _lib.check(L.od_nms(dl(tb), dl(ts), dl(tn), 0.5, max_out, dl(keep), dl(num), ws.data_ptr(), ws.numel(),
                            _lib.stream_ptr(tb.device)), "od_nms")
    _, names = trace(call)
    keep, num = host(keep), host(num)
    want = np.full((B, max_out), -1, np.int32)
    for b in range(B):
        w = oracle.nms(boxes[b, :nv[b]], scores[b, :nv[b]], max_out, 0.5)
        want[b, :w.shape[0]] = w
        assert num[b] == w.shape[0], (b, num[b], w.shape[0])
    assert np.array_equal(keep, want), "keep lists differ (padding included)"
    assert_written(keep, "keep_idx")
    assert_written(num, "num_kept")
    return names


def _topk_scores(rs, rows, cols):
    s = (np.round(rs.random_sample((rows, cols)) * 2048) / 2048).astype(f32)   # ties everywhere
    t = cols - 1 - (cols - 1) % C("kTileKeys")
    s[:, t::2] = s[:, t:t + 1]                                                    # ties in the last, partial tile
    s[:, -1] = s.max()                                                        # the largest score last
    return s


def run_topk(trace, rows, cols, k, s=None):
    _lib, L, dl = _L()
    rs = np.random.RandomState(rows * 31 + cols + k)
    if s is None:
        s = _topk_scores(rs, rows, cols)
    ts = cu(s)
    v, i = sent_f32((rows, k)), sent_i32((rows, k))

    def call():
        ws = poison(L.od_topk_workspace_bytes(rows, cols, k), ts.device)
        _lib.check(L.od_topk(dl(ts), k, dl(v), dl(i), ws.data_ptr(), ws.numel(), _lib.stream_ptr(ts.device)), "od_topk")
    _, names = trace(call)
    v, i = host(v), host(i)
    wv, wi = oracle.topk(s, k)
    assert np.array_equal(i, wi)
    assert_bits(v, wv, "values")
    assert np.array_equal(v.view(np.uint32), wv.view(np.uint32))
    assert_written(v, "values")
    assert_written(i, "indices")
    # independent: a stable sort on (-score, index) (no signed zeros or NaN in these rows)
    assert not np.isnan(s).any() and not ((s == 0) & np.signbit(s)).any()
    order = np.argsort(-s, axis=1, kind="stable")[:, :k]
    assert np.array_equal(i, order)
    return names


def _roi_maps(rs, B, D=256, sizes=(64, 32, 16, 8)):
    return [rs.random_sample((B, s, s, D)).astype(f32) for s in sizes]


def _edge_rois(rs, B, N):
    """rois_with_edge_cases with the hard rows moved into the last rows of the last image as well."""
    props = _synth.rois_log_uniform(rs, B, N, lo=4, hi=900)
    hard = _synth.rois_with_edge_cases(rs, 2, 13)[0]
    n = min(13, N)
    props[B - 1, N - n:] = hard[:n]
    if N > 30:
        props[0, :13] = hard
        props[B - 1, N - 20:N - 13] = 0                                           # zero padding next to the tail
    return props


def run_pyramid(trace, B, N, pool, order_ws=True):
    _lib, L, dl = _L()
    rs = np.random.RandomState(B * 1000 + N + pool[0])
    fmaps = _roi_maps(rs, B)
    props = _edge_rois(rs, B, N)
    fm, pr = [cu(f) for f in fmaps], cu(props)
    total = B * N
    out, lv = sent_f32((1, total, pool[0], pool[1], 256)), sent_i32((B, N))
    dev = pr.device
    zws = _lib.zeroed_workspace(L.od_pyramid_roi_align_workspace_bytes_n(total) if order_ws else
                                L.od_pyramid_roi_align_workspace_bytes(), dev)
    assert int(zws[:256].count_nonzero()) == 0
    ptrs = (ctypes.c_void_p * 4)(*[dl(f) for f in fm])

    def call():
        zws[256:].fill_(0xFF)                                                     # scratch after the ticket bytes
        _lib.check(L.od_pyramid_roi_align_forward_ws(ptrs, 4, 2, dl(pr), 1024, 1024, pool[0], pool[1], dl(out), dl(lv),
                                                     zws.data_ptr(), zws.numel(), _lib.stream_ptr(dev)),
                   "od_pyramid_roi_align_forward_ws")
    _, names = trace(call)
    got, glv = host(out), host(lv)
    assert int(zws[:256].count_nonzero()) == 0, "the ticket bytes were not left zeroed"
    want, wlv = oracle.pyramid_roi_align(fmaps, props, 1024, 1024, pool[0], pool[1])
    assert np.array_equal(glv, wlv)
    assert_bits(got, want, "pooled")
    assert_written(got[0], "pooled")
    assert_written(glv, "roi_level")
    return names, got, fmaps, props


def run_crop(trace, n, crop, D, check_f64):
    _lib, L, dl = _L()
    rs = np.random.RandomState(n * 13 + D + crop[0])
    img = rs.random_sample((3, 19, 23, D)).astype(f32)
    boxes = _synth.random_boxes(rs, n, flip=True)
    hard = np.array([[0, 0, 1, 1], [0.3, 0.3, 0.3, 0.3], [-0.2, -0.1, 0.5, 0.5], [0.5, 0.5, 1.3, 1.2],
                     [0.9, 0.8, 0.1, 0.2], [0, 0, 0, 0], [np.nan, 0.1, 0.5, 0.6]], f32)
    m = min(len(hard), n)
    boxes[n - m:] = hard[:m]                                                  # hard rows in the last CTA's bins
    bi = rs.randint(0, 3, n).astype(np.int32)
    skip = np.zeros(n, bool)
    if n >= 3:
        bi[n - 2], bi[0] = 3, -1                                             # out of range: crop left untouched
        skip[[0, n - 2]] = True
    ti, tbx, tbi = cu(img), cu(boxes), cu(bi)
    out = sent_f32((n, crop[0], crop[1], D))

    def call():
        _lib.check(L.od_crop_and_resize(dl(ti), dl(tbx), dl(tbi), crop[0], crop[1], 0.5, dl(out),
                                        _lib.stream_ptr(ti.device)), "od_crop_and_resize")
    _, names = trace(call)
    got = host(out)
    want = oracle.crop_and_resize(img, boxes, bi, crop[0], crop[1], extrapolation=0.5,
                                  out=np.full(got.shape, F_SENT, np.uint32).view(f32))
    assert_bits(got, want, "crops")
    assert_written(got, "crops", untouched=skip)
    if check_f64:
        w64, ok = crop_and_resize_f64(img, boxes, bi, *crop, extrapolation=0.5)
        ok = ok & ~skip[:, None, None] & ~np.isnan(boxes).any(1)[:, None, None]
        _assert_close_f64(got, w64, ok, f"crop n={n}")
    return names


def run_targets(trace, N, G, R=None, seed=0):
    _lib, L, dl = _L()

    class Cf(Conf):
        pass
    conf = Cf()
    R = R or conf.MRCNN_TRAIN_ROIS_PER_IMAGE
    rs = np.random.RandomState(N * 3 + G + R + seed)
    B = 2
    n_pad = max(1, N // 10)
    if G > N - n_pad:                                                          # many GT boxes, most of them valid
        from test_gpu_dispatch import _many_gt_inputs
        props, cls, gt, pp, pn = _many_gt_inputs(rs, B, N, G, n_pad=n_pad)
    else:
        props, cls, gt, pp, pn = _synth.target_inputs(rs, B, N, G, n_pad=n_pad)
    # hard rows at the end of the valid proposals: duplicates of a GT box, a zero row inside, a flipped box
    for b in range(B):
        e = N - n_pad
        props[b, e - 1] = gt[b, 0]
        props[b, e - 2] = props[b, e - 3]
        if e > 5:
            props[b, e - 4] = 0
            props[b, e - 5] = props[b, e - 5][[2, 3, 0, 1]]
    t = {k: cu(v) for k, v in dict(props=props, cls=cls, gt=gt, pp=pp, pn=pn).items()}
    rois, rcls, deltas = sent_f32((B, R, 4)), sent_i32((B, R)), sent_f32((B, R, 4))
    d = dict(iou=sent_f32((B, N, G)), roi_iou_max=sent_f32((B, N)), pos_indices=sent_i32((B, N)),
             neg_indices=sent_i32((B, N)), counts=sent_i32((B, 6)), sampled_pos=sent_i32((B, R)),
             sampled_neg=sent_i32((B, R)), gt_assignment=sent_i32((B, R)))
    dbg = _lib.TargetDebug(*[dl(d[k]) for k, _ in _lib.TargetDebug._fields_])
    params = _lib.TargetParams(R, (ctypes.c_float * 4)(*conf.BBOX_STD_DEV), 28, 28, 1, 1)
    dev = rois.device

    def call():
        ws = poison(L.od_detection_target_workspace_bytes(B, N, G), dev)
        _lib.check(L.od_detection_target_forward(dl(t["props"]), dl(t["cls"]), dl(t["gt"]), dl(t["pp"]), dl(t["pn"]),
                                                 ctypes.byref(params), dl(rois), dl(rcls), dl(deltas), None, None,
                                                 ctypes.byref(dbg), ws.data_ptr(), ws.numel(), _lib.stream_ptr(dev)),
                   "od_detection_target_forward")
    _, names = trace(call)
    rois, rcls, deltas = host(rois), host(rcls), host(deltas)
    d = {k: host(v) for k, v in d.items()}
    for b in range(B):
        w_rois, w_cls, w_deltas, wd = oracle.detection_targets(props[b], cls[b], gt[b], pp[b], pn[b], R, conf.BBOX_STD_DEV)
        assert np.array_equal(d["counts"][b], wd["counts"]), (b, d["counts"][b], wd["counts"])
        for k in ("pos_indices", "neg_indices", "sampled_pos", "sampled_neg", "gt_assignment"):
            assert np.array_equal(d[k][b], wd[k]), k
        n_prop, n_gt = wd["counts"][:2]
        assert_bits(d["iou"][b][:n_prop, :n_gt], wd["iou"][:n_prop, :n_gt], "iou")
        assert_bits(d["roi_iou_max"][b][:n_prop], wd["roi_iou_max"][:n_prop], "iou max")
        assert_bits(rois[b], w_rois, "rois")
        assert np.array_equal(rcls[b], w_cls[0])
        assert_bits(deltas[b], w_deltas, "deltas")
    for k, a in (("rois", rois), ("roi_gt_class_ids", rcls), ("roi_gt_box_deltas", deltas)):
        assert_written(a, k)
    for k in ("pos_indices", "neg_indices", "counts", "sampled_pos", "sampled_neg", "gt_assignment"):
        assert_written(d[k], k)
    return names, d


def _det_inputs(rs, B, N, C, kept=None):
    props = _synth.rois_log_uniform(rs, B, N)
    probs, bbox = _synth.head_outputs(rs, B, N, C, boosted=0.6)
    if kept is not None:
        # exactly `kept` rows per image pass DETECTION_MIN_THRESHOLD (0.7) with a foreground argmax: the others are
        # background-argmax rows or foreground rows at 0.7 exactly (not > 0.7)
        probs = np.full((B, N, C), 0.1 / (C - 1), f32)
        for b in range(B):
            rows = np.sort(rs.choice(N, kept, replace=False)) if b == 0 else np.arange(N - kept, N)
            cls = rs.randint(1, C, N)
            probs[b, np.arange(N), 0] = 0.9
            probs[b, rows, 0] = 0.01
            probs[b, rows, cls[rows]] = rs.uniform(0.71, 0.99, kept).astype(f32)
            at = np.setdiff1d(np.arange(N), rows)[:50]
            probs[b, at, 0] = 0.0
            probs[b, at, cls[at]] = f32(0.7)
    else:
        probs[1, 40:, 0] = 1.0                                                # image 1: few rows to keep, padded output
    if kept is not None:                                                      # image 1: one box per class survives NMS
        rows = np.arange(N - kept, N)
        props[1, rows] = props[1, 0]
        bbox[1, rows] = 0
    props[-1, N - 3:] = 0                                                     # zero padded rows in the tail
    props[-1, N - 5] = props[-1, N - 6]                                      # a duplicate ROI
    return props, probs, bbox


def run_detection(trace, N, kept=None, C=5, dts=(F32, F32)):
    """dts: the dtypes of mrcnn_class_probs and mrcnn_bbox (bf16 inputs hold bf16 values; the oracle sees them widened)."""
    _lib, L, dl = _L()
    conf = Conf()
    rs = np.random.RandomState(N * 11 + (kept or 0))
    B, M = 2, conf.DETECTION_POST_NMS_INSTANCES
    props, probs, bbox = _det_inputs(rs, B, N, C, kept)
    (probs, bbox), (tpr, tbb) = head_inputs((probs, bbox), dts, dts)
    win_px = np.array([[131, 0, 893, 1024], [0, 0, 1024, 1024]], np.int32)
    win = oracle.norm_boxes(win_px, [1024, 1024]).astype(f32)
    tp, tw = cu(props), cu(win)
    det = sent_f32((B, M, 6))
    d = dict(class_ids=sent_i32((B, N)), class_scores=sent_f32((B, N)), refined_proposals=sent_f32((B, N, 4)),
             clipped_proposals=sent_f32((B, N, 4)), keep_mask=sent_i32((B, N)), nms_keep_mask=sent_i32((B, N)))
    dbg = _lib.DetectionDebug(*[dl(d[k]) if k in d else None for k, _ in _lib.DetectionDebug._fields_])
    params = _lib.DetectionParams((ctypes.c_float * 4)(*conf.BBOX_STD_DEV), conf.DETECTION_MIN_THRESHOLD,
                                  conf.DETECTION_NMS_THRESHOLD, M)
    dev = tp.device

    def call():
        ws = poison(L.od_detection_workspace_bytes(B, N, C), dev)
        _lib.check(L.od_detection_forward(dl(tp), dl(tpr), dl(tbb), dl(tw), ctypes.byref(params), dl(det),
                                          ctypes.byref(dbg), ws.data_ptr(), ws.numel(), _lib.stream_ptr(dev)),
                   "od_detection_forward")
    _, names = trace(call)
    got = host(det)
    d = {k: host(v) for k, v in d.items()}
    want, wd = oracle.detection_forward(props, probs, bbox, win, conf.BBOX_STD_DEV, conf.DETECTION_MIN_THRESHOLD,
                                        conf.DETECTION_NMS_THRESHOLD, M, debug=True)
    assert np.array_equal(d["class_ids"], wd["class_ids"])
    assert_bits(d["class_scores"], wd["class_scores"], "class_scores")
    assert_bits(d["refined_proposals"], wd["refined_proposals"], "refined")
    assert_bits(d["clipped_proposals"], wd["clipped_proposals"], "clipped")
    assert np.array_equal(d["keep_mask"], wd["keep_mask"])
    assert np.array_equal(d["nms_keep_mask"], wd["nms_keep_mask"])
    assert_bits(got, want, "detections")
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    assert_written(got, "detections")
    for k, a in d.items():
        assert_written(a, k)
    if kept is not None:
        assert (wd["keep_mask"].sum(1) == kept).all()
    assert (got[1, :, 4] == 0).any(), "image 1 must end in zero padding"
    return names, got


def run_rpn_loss(trace, A, dts=(F32, F32), vals=None):
    """dts: the dtypes of rpn_class_logits and rpn_pred_box; vals (default dts): the inputs that hold bf16 values.
    Returns the kernel names and the outputs (losses, pred_box_pos, num_pos)."""
    _lib, L, dl = _L()
    rs = np.random.RandomState(A)
    B, T = 2, 256
    tc = rs.choice([-1, 0, 1], size=(B, A), p=[.3, .6, .1]).astype(np.int32)
    tc[:, A - 1], tc[:, A - 2] = 1, -1                                        # the last anchor of the last chunk counts
    lg = rs.normal(0, 2, (B, A, 2)).astype(f32)
    tb = rs.normal(0, 1, (B, T, 4)).astype(f32)
    pb = rs.normal(0, 1, (B, A, 4)).astype(f32)
    (lg, pb), (tlg, tpb) = head_inputs((lg, pb), dts, vals or dts)
    t = [cu(tc), tlg, cu(tb), tpb]
    P = int((tc == 1).sum())
    out, pos, num = sent_f32((2,)), sent_f32((P, 4)), sent_i32((1,))

    def call():
        ws = poison(L.od_rpn_loss_workspace_bytes(B, A), t[0].device)
        _lib.check(L.od_rpn_loss_forward(*[dl(x) for x in t], dl(out), dl(pos), dl(num), ws.data_ptr(), ws.numel(),
                                         _lib.stream_ptr(t[0].device)), "od_rpn_loss_forward")
    _, names = trace(call)
    out, pos, num = host(out), host(pos), host(num)
    wc, wb, wpos = oracle.rpn_losses(tc, lg, tb, pb)
    assert np.isclose(out[0], wc, rtol=1e-6) and np.isclose(out[1], wb, rtol=1e-6), (out, wc, wb)
    assert num[0] == P and np.array_equal(pos, wpos)
    assert_written(out, "losses")
    assert_written(pos, "pred_box_pos")
    assert_written(num, "num_pos")
    return names, (out, pos, num)


def run_mrcnn_loss(trace, BR, dts=(F32, F32), vals=None):
    """dts: the dtypes of mrcnn_pred_logits and mrcnn_pred_box; vals (default dts): the inputs that hold bf16 values.
    Returns the kernel names and the outputs (losses, pred_active)."""
    _lib, L, dl = _L()
    rs = np.random.RandomState(BR)
    B, R, C = 1, BR, 7
    ids = np.zeros((B, R), np.int32)
    ids[:, rs.random_sample(R) < 0.3] = rs.randint(1, C)
    ids[:, R - 1] = 2                                                         # the last ROI of the last pass is positive
    lg = rs.normal(0, 2, (B, R, C)).astype(f32)
    act = np.ones((B, C), f32)
    act[0, 3] = 0
    tb = rs.random_sample((B, R, 4)).astype(f32)
    pb = rs.random_sample((B, R, C, 4)).astype(f32)
    (lg, pb), (tlg, tpb) = head_inputs((lg, pb), dts, vals or dts)
    t = [cu(ids), tlg, cu(act), cu(tb), tpb]
    out, pa = sent_f32((2,)), sent_f32((B, R))

    def call():
        _lib.check(L.od_mrcnn_loss_forward(*[dl(x) for x in t], dl(out), dl(pa), _lib.stream_ptr(t[0].device)),
                   "od_mrcnn_loss_forward")
    _, names = trace(call)
    out, pa = host(out), host(pa)
    w_pa, w_c, w_b = oracle.mrcnn_losses(ids, lg, act, tb, pb)
    assert np.array_equal(pa, w_pa)
    assert np.isclose(out[0], w_c, rtol=1e-6) and np.isclose(out[1], w_b, rtol=1e-6), (out, w_c, w_b)
    assert_written(out, "losses")
    assert_written(pa, "pred_active")
    return names, (out, pa)


def run_rpn_targets(trace, A, G):
    _lib, L, dl = _L()
    rs = np.random.RandomState(A + 17 * G)
    B, T = 2, 64
    c = rs.uniform(0, 512, (A, 2))
    hw = rs.uniform(16, 128, (A, 2))
    anc = np.round(np.concatenate([c - hw / 2, c + hw / 2], 1))
    cnt = np.array([G, max(1, G - 5)], np.int32)
    gt = np.zeros((B, G, 4))
    for b in range(B):
        src = np.concatenate([rs.choice(A - 8, cnt[b] - 1, replace=False), [A - 1]])   # one GT on the last anchor
        gt[b, :cnt[b]] = anc[src] + np.round(rs.normal(0, 2, (cnt[b], 4)))
        bad = (gt[b, :, 2] <= gt[b, :, 0] + 1) | (gt[b, :, 3] <= gt[b, :, 1] + 1)
        gt[b, bad] = [100, 100, 164, 164]
    pp = np.stack([rs.permutation(A) for _ in range(B)]).astype(np.int32)
    pn = np.stack([rs.permutation(A) for _ in range(B)]).astype(np.int32)
    ta, tg, tcnt, tpp, tpn = cu(anc), cu(gt), cu(cnt), cu(pp), cu(pn)
    sd = [0.1, 0.1, 0.2, 0.2]
    params = _lib.RpnTargetParams(T, (ctypes.c_double * 4)(*sd))
    cls, bbox, pos, counts = sent_i32((B, A)), sent_f64((B, T, 4)), sent_f64((B, T, 4)), sent_i32((B, 4))

    def call():
        ws = poison(L.od_rpn_target_workspace_bytes(B, A, G), ta.device)
        _lib.check(L.od_rpn_target_forward(dl(ta), dl(tg), dl(tcnt), dl(tpp), dl(tpn), ctypes.byref(params), dl(cls),
                                           dl(bbox), dl(pos), dl(counts), ws.data_ptr(), ws.numel(),
                                           _lib.stream_ptr(ta.device)), "od_rpn_target_forward")
    _, names = trace(call)
    cls, bbox, pos, counts = host(cls), host(bbox), host(pos), host(counts)
    for b in range(B):
        w_pos, w_cls, w_bbox, w_counts = oracle.rpn_targets(anc, gt[b, :cnt[b]], pp[b], pn[b], T, sd)
        assert np.array_equal(counts[b], w_counts), (counts[b], w_counts)
        assert np.array_equal(cls[b], w_cls)
        n = w_counts[2]
        assert np.array_equal(pos[b, :n], w_pos) and not pos[b, n:].any()
        assert np.allclose(bbox[b], w_bbox, rtol=1e-13, atol=0)
    for k, a in (("rpn_target_class", cls), ("rpn_target_bbox", bbox), ("positive_anchors", pos), ("counts", counts)):
        assert_written(a, k)
    return names


def _crop_rois_f64(fmaps, props, pool):
    from test_gpu_dispatch import _pyramid_f64
    return _pyramid_f64(fmaps, props, pool)


# ------------------------------------------------------------------ the GPU cases
@pytest.mark.gpu
@pytest.mark.parametrize("name,value", CASES)
def test_boundary(_cuda, kernel_trace, name, value):
    b = BY_NAME[name]
    v = resolve(value)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    names = None
    if name in ("nms_ring_slots", "nms_staged_limit"):
        names = run_nms(kernel_trace, v, v)
    elif name == "nms_two_rounds":
        names = run_nms(kernel_trace, 6000, v)
        mask = sum(1 for n in names if "nms_mask_kernel<true>(" in _flat(n))
        assert mask == (2 if nms_two_rounds(6000, v) else 1), f"{mask} nms_mask_kernel launches at max_out = {v}"
    elif name == "topk_merge_smem":
        names = run_topk(kernel_trace, 2, 8000, v)
    elif name == "topk_tile":
        names = run_topk(kernel_trace, 2, 5000, v)
    elif name == "topk_merge_max":
        names = run_topk(kernel_trace, 1, 20000, v)
    elif name == "topk_index_bits":
        names = run_topk(kernel_trace, 2, v, 1000)
    elif name == "topk_cand_capacity":
        # 500 keys above the threshold bucket, then `v` keys of [0.5, 0.5625) (one 12-bit digit), the rest below
        rs = np.random.RandomState(v)
        cols = 40000
        s = rs.uniform(0.01, 0.4, (2, cols)).astype(f32)
        for r in range(2):
            at = (rs.permutation(cols) if r == 0 else                          # row 1: the bucket at the row's end
                  np.concatenate([rs.permutation(cols - v)[:500], np.arange(cols - v, cols)]))
            s[r, at[:500]] = rs.uniform(0.6, 0.9, 500).astype(f32)
            s[r, at[500:500 + v]] = (0.5 + np.floor(rs.uniform(0, 0.0624, v) * 4096) / 4096).astype(f32)
        s[1, -3:] = s[1, -4]                                                    # ties in the bucket, at the row's end
        assert (((s >= 0.5) & (s < 0.5625)).sum(1) == v).all()
        names = run_topk(kernel_trace, 2, cols, 1000, s)
    elif name == "topk_blocks_cols":
        names = run_topk(kernel_trace, 2, v, 1000)
    elif name == "topk_blocks_rows":
        names = run_topk(kernel_trace, v, 5000, 1000)
    elif name == "crop_rows_grid":
        names = run_crop(kernel_trace, v, (14, 14), 256, check_f64=v <= 160)
    elif name == "roi_align_mask_branch":
        names, got, fmaps, props = run_pyramid(kernel_trace, 1, v, [14, 14], order_ws=False)
        want, ok = _crop_rois_f64(fmaps, props, [14, 14])
        ok &= ~np.isnan(props).any(-1).reshape(-1)[:, None, None]
        _assert_close_f64(got[0], want, ok, f"pyramid n={v}")
    elif name == "roi_order_n":
        names = run_pyramid(kernel_trace, 1, v, [14, 14])[0]
    elif name == "roi_order_per_image":
        names = run_pyramid(kernel_trace, 1, v, [7, 7])[0]
    elif name == "crop_bins_32":
        names = run_crop(kernel_trace, v, (1, 1), 64, check_f64=True)
    elif name == "crop_bins_512":
        names = run_crop(kernel_trace, v, (1, 1), 8, check_f64=True)
    elif name == "targets_gt_smem":
        names, d = run_targets(kernel_trace, 300, v)
        assert (d["counts"][:, 1] > v - 400).all()                               # valid GT rows fill most of the table
    elif name in ("targets_iou_rows", "targets_compaction"):
        names, _ = run_targets(kernel_trace, v, 20)
    elif name == "targets_rois":
        names, d = run_targets(kernel_trace, 3200, 60, R=v)
        assert (d["counts"][:, 5] > 0).all()
    elif name in ("det_rank_tile", "det_rank_vs_sort", "det_scan_short_rows"):
        names, _ = run_detection(kernel_trace, v)
    elif name == "det_finalize_kept":
        names, got = run_detection(kernel_trace, 2048, kept=v)
    elif name == "rpn_loss_chunk":
        names, _ = run_rpn_loss(kernel_trace, v)
    elif name == "mrcnn_loss_cta":
        names, _ = run_mrcnn_loss(kernel_trace, v)
    elif name == "rpn_target_chunk":
        names = run_rpn_targets(kernel_trace, v, 12)
    elif name == "rpn_target_fused_gt":
        names = run_rpn_targets(kernel_trace, 3000, v)
    else:
        raise AssertionError(f"no runner for {name}")
    if b.kernels is not None:
        must, must_not = b.kernels(v, sms)
        assert_launched(names, must=must, must_not=must_not)
