// targets.cu — DetectionTargetLayer: BuildDetectionTargets.build_detection_target
// (data_processor.py:512-652) with get_iou_tf (:473-510) and box_refinement_tf (:443-471), batched.
//
// Two kernels. detection_iou_kernel (8 CTAs of 256 proposals per image at N = 2000): GT boxes sit in shared memory and
// each thread reduces one proposal row of the N x G IoU matrix to (max, first argmax); the matrix is never materialised
// (unless the debug tensor is requested). The zero-padding strip of the proposals is a stable compaction whose base per
// CTA is a count over the rows in front of it. detection_target_kernel (one CTA per image) does the sequential part:
// pos/neg index lists are stable block compactions (ascending index == tf.where order). tf.random_shuffle
// (:587,:597) is replaced by explicit permutation inputs: the shuffled list is list[q] for q in perm (in
// order) with q < len(list).
#include "common.cuh"

namespace od {

constexpr int kTgtThreads = 1024;
constexpr int kIouThreads = 256;

struct TargetDebugPtrs {
  float* iou;              // [B,N,G]
  float* roi_iou_max;      // [B,N]
  int32_t* pos_indices;    // [B,N]
  int32_t* neg_indices;    // [B,N]
  int32_t* counts;         // [B,6]
  int32_t* sampled_pos;    // [B,R]
  int32_t* sampled_neg;    // [B,R]
  int32_t* gt_assignment;  // [B,R]
};

// get_iou_tf: no canonicalisation, no area guard.
__device__ __forceinline__ float target_iou(float4 p, float4 g) {
  const float p_area = (p.z - p.x) * (p.w - p.y);
  const float g_area = (g.z - g.x) * (g.w - g.y);
  const float iy1 = f_max(p.x, g.x), ix1 = f_max(p.y, g.y);
  const float iy2 = f_min(p.z, g.z), ix2 = f_min(p.w, g.w);
  const float inter = f_max(iy2 - iy1, 0.0f) * f_max(ix2 - ix1, 0.0f);
  return inter / ((p_area + g_area) - inter);
}

// box_refinement_tf followed by "/= stddev".
__device__ __forceinline__ float4 refine_box(float4 box, float4 gt, float4 sd) {
  const float height = box.z - box.x;
  const float width = box.w - box.y;
  const float center_y = box.x + 0.5f * height;
  const float center_x = box.y + 0.5f * width;
  const float gt_height = gt.z - gt.x;
  const float gt_width = gt.w - gt.y;
  const float gt_center_y = gt.x + 0.5f * gt_height;
  const float gt_center_x = gt.y + 0.5f * gt_width;
  return make_float4(((gt_center_y - center_y) / height) / sd.x, ((gt_center_x - center_x) / width) / sd.y,
                     f_log(gt_height / height) / sd.z, f_log(gt_width / width) / sd.w);
}

// Stable compaction of {i in [0,n) : pred(i)}; emit(i, rank) is called for every selected i. Returns the
// count. All threads of the CTA must call it; `scratch` holds 34 ints.
template <typename Pred, typename Emit>
__device__ int block_stable_compact(int n, Pred pred, Emit emit, int* scratch) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nwarps = blockDim.x >> 5;
  int base = 0;
  for (int t0 = 0; t0 < n; t0 += blockDim.x) {
    const int i = t0 + tid;
    const bool p = (i < n) && pred(i);
    const uint32_t bal = __ballot_sync(0xffffffffu, p);
    if (lane == 0) scratch[warp] = __popc(bal);
    __syncthreads();
    int off = 0, total = 0;
    for (int w = 0; w < nwarps; ++w) {
      const int c = scratch[w];
      if (w < warp) off += c;
      total += c;
    }
    if (p) emit(i, base + off + __popc(bal & ((1u << lane) - 1u)));
    base += total;
    __syncthreads();
  }
  return base;
}

__device__ __forceinline__ bool prop_nonzero(float4 p) {
  return (((fabsf(p.x) + fabsf(p.y)) + fabsf(p.z)) + fabsf(p.w)) != 0.0f;
}

// (1) strip zero padding (:564-571) and (2) IoU rows -> max / first argmax (:576-579, :610) for proposals
// [blockIdx.x * 64, +64) of image blockIdx.y. Four lanes share a row: lane part p takes GT boxes p, p+4, ... and the
// quad combines (greater value wins, equal values keep the smaller GT index = the first arg-max of the serial scan).
// Outputs are indexed by the COMPACTED proposal index.
constexpr int kIouRows = kIouThreads / 4;
__global__ void __launch_bounds__(kIouThreads)
detection_iou_kernel(const float4* __restrict__ proposals, const int32_t* __restrict__ gt_class_ids,
                     const float4* __restrict__ gt_boxes, int N, int G, int32_t* __restrict__ ws_i32,
                     float* __restrict__ ws_f32, int32_t* __restrict__ n_prop_out, TargetDebugPtrs dbg) {
  pdl_prologue();
  extern __shared__ float4 s_gt[];                        // [G] compacted GT boxes
  __shared__ int scratch[40];
  __shared__ int s_base, s_rank[kIouRows], s_cnt[2];
  const int b = blockIdx.y, tid = threadIdx.x, r0 = blockIdx.x * kIouRows;
  const float4* prop = proposals + (int64_t)b * N;
  const int32_t* gcls = gt_class_ids + (int64_t)b * G;
  const float4* gbox = gt_boxes + (int64_t)b * G;
  int32_t* prop_src = ws_i32 + (int64_t)b * 4 * N;
  int32_t* iou_arg = prop_src + N;
  float* iou_max = ws_f32 + (int64_t)b * N;
  if (tid == 0) s_base = 0;
  __syncthreads();
  const int n_gt = block_stable_compact(
      G, [&](int j) { return gcls[j] != 0; }, [&](int j, int r) { s_gt[r] = gbox[j]; }, scratch);
  // non-zero rows in front of this CTA's slice
  int cnt = 0;
  for (int i = tid; i < r0; i += kIouThreads) cnt += prop_nonzero(prop[i]) ? 1 : 0;
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, d);
  if ((tid & 31) == 0 && cnt) atomicAdd(&s_base, cnt);
  // stable rank of this slice's non-zero rows (threads 0..63 = two warps)
  if (tid < kIouRows) {
    const bool nz = (r0 + tid < N) && prop_nonzero(prop[r0 + tid]);
    const uint32_t bal = __ballot_sync(0xffffffffu, nz);
    if ((tid & 31) == 0) s_cnt[tid >> 5] = __popc(bal);
    s_rank[tid] = nz ? __popc(bal & ((1u << (tid & 31)) - 1u)) : -1;
  }
  __syncthreads();
  const int k = tid >> 2, part = tid & 3;
  int rank = s_rank[k];
  if (rank >= 0 && k >= 32) rank += s_cnt[0];
  const int i = s_base + rank;                            // compacted index (valid when rank >= 0)
  const bool row = rank >= 0;                             // uniform per quad
  float best = -INFINITY;
  int arg = 0;
  if (row) {
    OD_DBG_IDX(i, N);
    const float4 p = prop[r0 + k];
    for (int j = part; j < n_gt; j += 4) {
      const float v = target_iou(p, s_gt[j]);
      if (dbg.iou) dbg.iou[((int64_t)b * N + i) * G + j] = v;
      if (v > best) {
        best = v;
        arg = j;
      }
    }
    if (best == -INFINITY) arg = 0;                       // nothing selected: the serial scan leaves arg at 0
  }
#pragma unroll
  for (int d = 1; d < 4; d <<= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, best, d);
    const int oa = __shfl_xor_sync(0xffffffffu, arg, d);
    if (ov > best || (ov == best && oa < arg)) {
      best = ov;
      arg = oa;
    }
  }
  if (row && part == 0) {
    prop_src[i] = r0 + k;
    iou_max[i] = best;
    iou_arg[i] = arg;
    if (dbg.roi_iou_max) dbg.roi_iou_max[(int64_t)b * N + i] = best;
  }
  if (tid == 0 && r0 + kIouRows >= N) n_prop_out[b] = s_base + s_cnt[0] + s_cnt[1];
}

__global__ void __launch_bounds__(kTgtThreads)
detection_target_kernel(const float4* __restrict__ proposals, const int32_t* __restrict__ gt_class_ids,
                        const float4* __restrict__ gt_boxes, const int32_t* __restrict__ perm_pos,
                        const int32_t* __restrict__ perm_neg, int N, int G, int R, float4 stddev,
                        float4* __restrict__ rois, int32_t* __restrict__ roi_cls, float4* __restrict__ roi_deltas,
                        int32_t* __restrict__ ws_i32, float* __restrict__ ws_f32, const int32_t* __restrict__ n_prop_in,
                        int32_t* __restrict__ mask_src, TargetDebugPtrs dbg) {
  pdl_prologue();
  extern __shared__ int32_t s_gt_src[];                   // [G] original GT row of compacted j
  __shared__ int scratch[40];
  const int b = blockIdx.x, tid = threadIdx.x;
  const float4* prop = proposals + (int64_t)b * N;
  const int32_t* gcls = gt_class_ids + (int64_t)b * G;
  const float4* gbox = gt_boxes + (int64_t)b * G;
  // per-image scratch in global memory: prop_src | arg | pos_list | neg_list (int32) and iou_max (f32)
  int32_t* prop_src = ws_i32 + (int64_t)b * 4 * N;
  int32_t* iou_arg = prop_src + N;
  int32_t* pos_list = iou_arg + N;
  int32_t* neg_list = pos_list + N;
  float* iou_max = ws_f32 + (int64_t)b * N;
  (void)prop_src;

  const int n_gt = block_stable_compact(
      G, [&](int j) { return gcls[j] != 0; }, [&](int j, int r) { s_gt_src[r] = j; }, scratch);
  const int n_prop = n_prop_in[b];
  __syncthreads();

  // (3) where(max >= 0.5) / where(max < 0.5), ascending (:582-583)
  const int n_pos = block_stable_compact(
      n_prop, [&](int i) { return iou_max[i] >= 0.5f; }, [&](int i, int r) { pos_list[r] = i; }, scratch);
  const int n_neg = block_stable_compact(
      n_prop, [&](int i) { return iou_max[i] < 0.5f; }, [&](int i, int r) { neg_list[r] = i; }, scratch);
  __syncthreads();
  if (dbg.pos_indices)
    for (int i = tid; i < N; i += kTgtThreads) dbg.pos_indices[(int64_t)b * N + i] = (i < n_pos) ? pos_list[i] : -1;
  if (dbg.neg_indices)
    for (int i = tid; i < N; i += kTgtThreads) dbg.neg_indices[(int64_t)b * N + i] = (i < n_neg) ? neg_list[i] : -1;

  // (4) counts (:586-594), fp32 arithmetic with truncation
  const int num_pos_inst = (int)((double)R * 0.33);
  const int pos_count = min(n_pos, num_pos_inst);
  const float inv = (float)(1.0 / 0.33);
  int neg_cnt = f_to_i32_x86(inv * (float)pos_count) - pos_count;
  neg_cnt = max(neg_cnt, 0);
  const int neg_count = min(min(n_neg, neg_cnt), R - pos_count);  // host guarantees the last bound never binds
  if (dbg.counts && tid == 0) {
    int32_t* c = dbg.counts + (int64_t)b * 6;
    c[0] = n_prop; c[1] = n_gt; c[2] = n_pos; c[3] = n_neg; c[4] = pos_count; c[5] = neg_count;
  }

  // (8) zero padding first, sampled rows overwrite below after a barrier
  float4* o_rois = rois + (int64_t)b * R;
  int32_t* o_cls = roi_cls + (int64_t)b * R;
  float4* o_del = roi_deltas + (int64_t)b * R;
  const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int t = tid; t < R; t += kTgtThreads) {
    if (t >= pos_count + neg_count) o_rois[t] = z4;
    if (t >= pos_count) {
      o_cls[t] = 0;
      o_del[t] = z4;
    }
    if (mask_src) mask_src[(int64_t)b * R + t] = -1;
    if (dbg.sampled_pos) dbg.sampled_pos[(int64_t)b * R + t] = -1;
    if (dbg.sampled_neg) dbg.sampled_neg[(int64_t)b * R + t] = -1;
    if (dbg.gt_assignment) dbg.gt_assignment[(int64_t)b * R + t] = -1;
  }
  __syncthreads();

  // (5)-(7) shuffled sampling, gather from the UN-compacted proposals (:600-616)
  const int32_t* pp = perm_pos + (int64_t)b * N;
  const int32_t* pn = perm_neg + (int64_t)b * N;
  block_stable_compact(
      N,
      [&](int t) {
        const int q = pp[t];
        return q >= 0 && q < n_pos;
      },
      [&](int t, int r) {
        if (r >= pos_count) return;
        const int idx = pos_list[pp[t]];
        OD_DBG_IDX(idx, N);
        const float4 box = prop[idx];
        const int a = iou_arg[idx];
        OD_DBG_IDX(a, G);
        const int g = s_gt_src[a];
        OD_DBG_IDX(g, G);
        OD_DBG_IDX(r, R);
        o_rois[r] = box;
        o_cls[r] = gcls[g];
        o_del[r] = refine_box(box, gbox[g], stddev);
        if (mask_src) mask_src[(int64_t)b * R + r] = g;
        if (dbg.sampled_pos) dbg.sampled_pos[(int64_t)b * R + r] = idx;
        if (dbg.gt_assignment) dbg.gt_assignment[(int64_t)b * R + r] = a;
      },
      scratch);
  block_stable_compact(
      N,
      [&](int t) {
        const int q = pn[t];
        return q >= 0 && q < n_neg;
      },
      [&](int t, int r) {
        if (r >= neg_count) return;
        const int idx = neg_list[pn[t]];
        OD_DBG_IDX(idx, N);
        OD_DBG_IDX(pos_count + r, R);
        o_rois[pos_count + r] = prop[idx];
        if (dbg.sampled_neg) dbg.sampled_neg[(int64_t)b * R + r] = idx;
      },
      scratch);
}

// Mask targets (north-star extension; the reference prepares batch_gt_masks at data_processor.py:386,399 but never
// consumes them because its mask head is commented out, masking.py:1-67). Semantics restated from the model this
// file re-writes (matterport Mask_RCNN detection_targets_graph): for every sampled positive ROI
//   box = roi                                   (full-size masks), or
//   box = (roi - gt_box.y1x1y1x1) / (gt_h, gt_w, gt_h, gt_w)        (mini masks: ROI in the GT box's frame)
//   target = round(crop_and_resize(gt_mask[assigned GT], box, [mask_h, mask_w]))   round = half to even
// rows of non-positive ROIs are zero. One CTA per (roi slot, image); D = 1 channel, so plain scalar taps: 4 bytes for
// fp32 masks, 1 byte for uint8 and bool masks. A byte widens to fp32 exactly (bool 0 / 1, uint8 0..255), and everything
// after the load is the fp32 path, so a byte mask gives the fp32 call's targets on the widened mask bit for bit.
__device__ __forceinline__ float ldg_mask(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ldg_mask(const uint8_t* p) { return (float)__ldg(p); }

template <typename TMask>
__device__ __forceinline__ void mask_target_body(const float4* __restrict__ rois, const float4* __restrict__ gt_boxes,
                                                 const int32_t* __restrict__ mask_src, const TMask* __restrict__ gt_masks,
                                                 int R, int G, int Mh, int Mw, int hwg_layout, int use_mini_mask, int mh,
                                                 int mw, float* __restrict__ targets) {
  const int r = blockIdx.x, b = blockIdx.y;
  float* o = targets + ((int64_t)b * R + r) * mh * mw;
  const int g = mask_src[(int64_t)b * R + r];
  const int total = mh * mw;
  if (g < 0) {
    for (int e = threadIdx.x; e < total; e += blockDim.x) o[e] = 0.0f;
    return;
  }
  float4 box = rois[(int64_t)b * R + r];
  if (use_mini_mask) {
    const float4 gt = gt_boxes[(int64_t)b * G + g];
    const float gt_h = gt.z - gt.x, gt_w = gt.w - gt.y;
    box = make_float4((box.x - gt.x) / gt_h, (box.y - gt.y) / gt_w, (box.z - gt.x) / gt_h, (box.w - gt.y) / gt_w);
  }
  // element (y, x) of GT mask g: [B,G,Mh,Mw] or the reference's [B,Mh,Mw,G]
  const TMask* img = gt_masks + (int64_t)b * G * Mh * Mw + (hwg_layout ? (int64_t)g : (int64_t)g * Mh * Mw);
  const int64_t sy = hwg_layout ? (int64_t)Mw * G : Mw, sx = hwg_layout ? G : 1;
  const float Hm1 = (float)(Mh - 1), Wm1 = (float)(Mw - 1);
  const float hs = (mh > 1) ? (box.z - box.x) * Hm1 / (float)(mh - 1) : 0.0f;
  const float ws = (mw > 1) ? (box.w - box.y) * Wm1 / (float)(mw - 1) : 0.0f;
  for (int e = threadIdx.x; e < total; e += blockDim.x) {
    const int y = e / mw, x = e - y * mw;
    const float in_y = (mh > 1) ? box.x * Hm1 + (float)y * hs : (float)(0.5 * (double)(box.x + box.z) * (double)(Mh - 1));
    const float in_x = (mw > 1) ? box.y * Wm1 + (float)x * ws : (float)(0.5 * (double)(box.y + box.w) * (double)(Mw - 1));
    float v = 0.0f;   // extrapolation_value = 0
    if ((in_y >= 0.0f) && (in_y <= Hm1) && (in_x >= 0.0f) && (in_x <= Wm1)) {
      const float fy = floorf(in_y), fx = floorf(in_x);
      const int64_t top = (int64_t)fy, bot = (int64_t)ceilf(in_y), left = (int64_t)fx, right = (int64_t)ceilf(in_x);
      const float yl = in_y - fy, xl = in_x - fx;
      const float tl = ldg_mask(img + top * sy + left * sx), tr = ldg_mask(img + top * sy + right * sx);
      const float bl = ldg_mask(img + bot * sy + left * sx), br = ldg_mask(img + bot * sy + right * sx);
      const float t = tl + (tr - tl) * xl;
      const float bt = bl + (br - bl) * xl;
      v = t + (bt - t) * yl;
    }
    o[e] = rintf(v);
  }
}

__global__ void __launch_bounds__(256)
mask_target_kernel(const float4* __restrict__ rois, const float4* __restrict__ gt_boxes, const int32_t* __restrict__ mask_src,
                   const float* __restrict__ gt_masks, int R, int G, int Mh, int Mw, int hwg_layout, int use_mini_mask,
                   int mh, int mw, float* __restrict__ targets) {
  mask_target_body<float>(rois, gt_boxes, mask_src, gt_masks, R, G, Mh, Mw, hwg_layout, use_mini_mask, mh, mw, targets);
}
// uint8 and bool masks (TMask = uint8_t): the same body, an overload of the same name (the fp32 kernel above keeps its name)
template <typename TMask>
__global__ void __launch_bounds__(256)
mask_target_kernel(const float4* __restrict__ rois, const float4* __restrict__ gt_boxes, const int32_t* __restrict__ mask_src,
                   const TMask* __restrict__ gt_masks, int R, int G, int Mh, int Mw, int hwg_layout, int use_mini_mask,
                   int mh, int mw, float* __restrict__ targets) {
  mask_target_body<TMask>(rois, gt_boxes, mask_src, gt_masks, R, G, Mh, Mw, hwg_layout, use_mini_mask, mh, mw, targets);
}

}  // namespace od

using namespace od;

extern "C" {

size_t od_detection_target_workspace_bytes(int64_t batch, int64_t num_proposals, int64_t num_gt) {
  Workspace w(nullptr, 0);
  w.take<int32_t>((size_t)(batch * 4 * num_proposals));
  w.take<float>((size_t)(batch * num_proposals));
  w.take<int32_t>((size_t)(batch * 4096));   // GT row of every sampled positive (mask targets), R <= 4096
  w.take<int32_t>((size_t)batch);            // non-zero proposals per image
  return w.off + 256;
}

int od_detection_target_forward(const DLTensor* proposals, const DLTensor* gt_class_ids, const DLTensor* gt_boxes,
                                const DLTensor* perm_pos, const DLTensor* perm_neg, const od_target_params* params,
                                DLTensor* rois, DLTensor* roi_gt_class_ids, DLTensor* roi_gt_box_deltas,
                                const DLTensor* gt_masks, DLTensor* mask_targets, const od_target_debug* debug,
                                void* ws, size_t ws_bytes, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (!params) OD_FAIL(OD_ERR_NULL, "params is NULL");
  DeviceScope scope;
  OD_CHECK(check_tensor(proposals, "proposals", F32, {kAny, kAny, 4}, 16, scope));
  const int64_t B = proposals->shape[0], N = proposals->shape[1], R = params->rois_per_image;
  OD_CHECK(check_tensor(gt_class_ids, "gt_class_ids", I32, {B, kAny}, 4, scope));
  const int64_t G = gt_class_ids->shape[1];
  OD_CHECK(check_tensor(gt_boxes, "gt_boxes", F32, {B, G, 4}, 16, scope));
  OD_CHECK(check_tensor(perm_pos, "perm_pos", I32, {B, N}, 4, scope));
  OD_CHECK(check_tensor(perm_neg, "perm_neg", I32, {B, N}, 4, scope));
  OD_CHECK(check_tensor(rois, "rois", F32, {B, R, 4}, 16, scope));
  OD_CHECK(check_tensor(roi_gt_class_ids, "roi_gt_class_ids", I32, {B, R}, 4, scope));
  OD_CHECK(check_tensor(roi_gt_box_deltas, "roi_gt_box_deltas", F32, {B, R, 4}, 16, scope));
  if ((gt_masks == nullptr) != (mask_targets == nullptr)) OD_FAIL(OD_ERR_NULL, "gt_masks and mask_targets go together");
  int64_t Mh = 0, Mw = 0;
  const DType mask_dt = f32_or_byte(gt_masks);            // f32, u8 or bool; a byte mask is read one byte per element
  if (gt_masks) {
    const int mask_align = (mask_dt == F32) ? 4 : 1;
    if (params->mask_layout_hwg) OD_CHECK(check_tensor(gt_masks, "gt_masks", mask_dt, {B, kAny, kAny, G}, mask_align, scope));
    else OD_CHECK(check_tensor(gt_masks, "gt_masks", mask_dt, {B, G, kAny, kAny}, mask_align, scope));
    Mh = gt_masks->shape[params->mask_layout_hwg ? 1 : 2];
    Mw = gt_masks->shape[params->mask_layout_hwg ? 2 : 3];
    if (params->mask_h < 1 || params->mask_w < 1 || Mh < 1 || Mw < 1) OD_FAIL(OD_ERR_PARAM, "mask sizes must be positive");
    OD_CHECK(check_tensor(mask_targets, "mask_targets", F32, {B, R, params->mask_h, params->mask_w}, 4, scope));
    if (R > 4096) OD_FAIL(OD_ERR_PARAM, "mask targets support rois_per_image <= 4096");
  }
  if (G > 8192) OD_FAIL(OD_ERR_PARAM, "at most 8192 GT boxes per image");
  if (N >= (1 << 30)) OD_FAIL(OD_ERR_PARAM, "too many proposals");
  // pos_count + neg_count must fit R for every reachable pos_count (data_processor.py:586-594 arithmetic)
  {
    const int num_pos_inst = (int)((double)R * 0.33);
    const float inv = (float)(1.0 / 0.33);
    for (int p = 0; p <= num_pos_inst; ++p)
      if ((int)(inv * (float)p) > R) OD_FAIL(OD_ERR_PARAM, "rois_per_image=%lld cannot hold pos+neg samples", (long long)R);
  }
  od_target_debug dbg;
  memset(&dbg, 0, sizeof(dbg));
  if (debug) dbg = *debug;
  OD_CHECK(check_opt_tensor(dbg.iou, "debug.iou", F32, {B, N, G}, 4, scope));
  OD_CHECK(check_opt_tensor(dbg.roi_iou_max, "debug.roi_iou_max", F32, {B, N}, 4, scope));
  OD_CHECK(check_opt_tensor(dbg.pos_indices, "debug.pos_indices", I32, {B, N}, 4, scope));
  OD_CHECK(check_opt_tensor(dbg.neg_indices, "debug.neg_indices", I32, {B, N}, 4, scope));
  OD_CHECK(check_opt_tensor(dbg.counts, "debug.counts", I32, {B, 6}, 4, scope));
  OD_CHECK(check_opt_tensor(dbg.sampled_pos, "debug.sampled_pos", I32, {B, R}, 4, scope));
  OD_CHECK(check_opt_tensor(dbg.sampled_neg, "debug.sampled_neg", I32, {B, R}, 4, scope));
  OD_CHECK(check_opt_tensor(dbg.gt_assignment, "debug.gt_assignment", I32, {B, R}, 4, scope));
  if (B == 0 || R == 0) return OD_OK;
  if (!ws) OD_FAIL(OD_ERR_WORKSPACE, "workspace is NULL");
  Workspace w(ws, ws_bytes);
  int32_t* ws_i32 = w.take<int32_t>((size_t)(B * 4 * N));
  float* ws_f32 = w.take<float>((size_t)(B * N));
  int32_t* mask_src = w.take<int32_t>((size_t)(B * 4096));
  int32_t* n_prop = w.take<int32_t>((size_t)B);
  if (!w.ok()) OD_FAIL(OD_ERR_WORKSPACE, "workspace %zu < %zu bytes", ws_bytes, w.off);
  TargetDebugPtrs dp;
  dp.iou = dptr<float>(dbg.iou);
  dp.roi_iou_max = dptr<float>(dbg.roi_iou_max);
  dp.pos_indices = dptr<int32_t>(dbg.pos_indices);
  dp.neg_indices = dptr<int32_t>(dbg.neg_indices);
  dp.counts = dptr<int32_t>(dbg.counts);
  dp.sampled_pos = dptr<int32_t>(dbg.sampled_pos);
  dp.sampled_neg = dptr<int32_t>(dbg.sampled_neg);
  dp.gt_assignment = dptr<int32_t>(dbg.gt_assignment);
  const float4 sd = make_float4(params->bbox_stddev[0], params->bbox_stddev[1], params->bbox_stddev[2], params->bbox_stddev[3]);
  const size_t smem_iou = (size_t)(G > 0 ? G : 1) * sizeof(float4);      // <= 128 KiB at the G <= 8192 cap
  static const size_t iou_static = static_smem_bytes((const void*)detection_iou_kernel);
  if (smem_iou + iou_static > 48 * 1024)
    OD_CUDA(cudaFuncSetAttribute(detection_iou_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_iou));
  if (N > 0) {
    const dim3 grid((unsigned)((N + kIouRows - 1) / kIouRows), (unsigned)B);
    OD_CUDA(launch_pdl(detection_iou_kernel, grid, dim3(kIouThreads), smem_iou, st, dptr<float4>(proposals),
                       dptr<int32_t>(gt_class_ids), dptr<float4>(gt_boxes), (int)N, (int)G, ws_i32, ws_f32, n_prop, dp));
    OD_LAUNCH_CHECK("detection_iou_kernel");
  } else {
    OD_CUDA(cudaMemsetAsync(n_prop, 0, (size_t)B * sizeof(int32_t), st));
  }
  const size_t smem = (size_t)(G > 0 ? G : 1) * sizeof(int32_t);
  OD_CUDA(launch_pdl(detection_target_kernel, dim3((unsigned)B), dim3(kTgtThreads), smem, st,
      dptr<float4>(proposals), dptr<int32_t>(gt_class_ids), dptr<float4>(gt_boxes), dptr<int32_t>(perm_pos),
      dptr<int32_t>(perm_neg), (int)N, (int)G, (int)R, sd, dptr<float4>(rois), dptr<int32_t>(roi_gt_class_ids),
      dptr<float4>(roi_gt_box_deltas), ws_i32, ws_f32, (const int32_t*)n_prop, gt_masks ? mask_src : nullptr, dp));
  OD_LAUNCH_CHECK("detection_target_kernel");
  if (gt_masks && mask_dt != F32) {
    const dim3 grid((unsigned)R, (unsigned)B);
    mask_target_kernel<uint8_t><<<grid, 256, 0, st>>>(dptr<float4>(rois), dptr<float4>(gt_boxes), mask_src, dptr<uint8_t>(gt_masks),
                                                      (int)R, (int)G, (int)Mh, (int)Mw, params->mask_layout_hwg ? 1 : 0,
                                                      params->use_mini_mask ? 1 : 0, params->mask_h, params->mask_w,
                                                      dptr<float>(mask_targets));
    OD_LAUNCH_CHECK("mask_target_kernel<uint8_t>");
  } else if (gt_masks) {
    const dim3 grid((unsigned)R, (unsigned)B);
    mask_target_kernel<<<grid, 256, 0, st>>>(dptr<float4>(rois), dptr<float4>(gt_boxes), mask_src, dptr<float>(gt_masks), (int)R,
                                             (int)G, (int)Mh, (int)Mw, params->mask_layout_hwg ? 1 : 0,
                                             params->use_mini_mask ? 1 : 0, params->mask_h, params->mask_w,
                                             dptr<float>(mask_targets));
    OD_LAUNCH_CHECK("mask_target_kernel");
  }
  return OD_OK;
}

}  // extern "C"
