// losses.cu — forward values of the four head losses (MaskRCNN/building_blocks/loss_optimize.py:11-201), the
// consumers of the RPN targets and of the detection targets. SURVEY.md §8(f) rank 4.
//
//   rpn_class_loss  (:11-44)   anchors with target != 0 -> 2-way sparse softmax cross-entropy, mean (0 if none)
//   rpn_box_loss    (:47-87)   positive anchors in (image, anchor) order against the first rows of the zero-padded
//                              rpn_target_bbox of their image -> smooth-L1, mean over the elements (0 if none)
//   mrcnn_class_loss (:89-151) sparse softmax cross-entropy per ROI, weighted by the active flag (of image 0, as the
//                              reference gathers batch_active_class_ids[0]) of the PREDICTED class; sum / sum
//   mrcnn_box_loss  (:154-201) positive ROIs, predicted box of the target class, K.binary_crossentropy(target, output)
//                              — the reference's choice (not smooth-L1) is kept — mean (0 if none)
//
// Every per-element value is fp32 in the reference's operation order (exp/log rounded from fp64 like the rest of the
// library); the sums are accumulated in fp64 in a fixed order (deterministic, independent of the grid) and rounded to
// fp32 once, so they agree with TensorFlow's fp32 tree reductions to ~1e-7 relative rather than bit for bit.
#include "common.cuh"

namespace od {

constexpr int kLossThreads = 256;
constexpr int kLossWarps = kLossThreads / 32;
constexpr int kLossChunk = 4 * kLossThreads;

struct RpnLossPart {
  double ce_sum;    // cross-entropy over the non-neutral anchors of the chunk
  double box_sum;   // smooth-L1 over the positive anchors of the chunk (second pass)
  int32_t nz, pos, used, pad;
};

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// Sum over the CTA, warps combined in index order; every thread gets the result. scratch: kLossWarps elements.
template <typename T>
__device__ T cta_sum(T v, T* scratch) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
  __syncthreads();
  T r = 0;
  for (int w = 0; w < (int)(blockDim.x >> 5); ++w) r += scratch[w];
  return r;
}

// Pass 1: per 1024-anchor chunk, the cross-entropy sum and the counts of non-neutral / positive anchors.
__global__ void __launch_bounds__(kLossThreads)
rpn_loss_class_kernel(const int32_t* __restrict__ target, const float2* __restrict__ logits, int A, RpnLossPart* __restrict__ part) {
  __shared__ double sd[kLossWarps];
  __shared__ int si[kLossWarps];
  const int b = blockIdx.y, i0 = blockIdx.x * kLossChunk + 4 * threadIdx.x;
  double ce = 0.0;
  int nz = 0, pos = 0;
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const int i = i0 + u;
    if (i >= A) break;
    const int t = target[(int64_t)b * A + i];
    if (t == 0) continue;
    const float2 x = __ldg(&logits[(int64_t)b * A + i]);
    const float m = f_max(x.x, x.y);
    const float s = f_exp(x.x - m) + f_exp(x.y - m);
    ce += (double)(f_log(s) - (((t == 1) ? x.y : x.x) - m));   // label 1 = foreground (:31)
    ++nz;
    pos += (t == 1) ? 1 : 0;
  }
  const double ce_all = cta_sum(ce, sd);
  const int nz_all = cta_sum(nz, si);
  const int pos_all = cta_sum(pos, si);
  if (threadIdx.x == 0) {
    RpnLossPart p;
    p.ce_sum = ce_all;
    p.box_sum = 0.0;
    p.nz = nz_all;
    p.pos = pos_all;
    p.used = 0;
    p.pad = 0;
    part[(int64_t)b * gridDim.x + blockIdx.x] = p;
  }
}

// Pass 2: the r-th positive anchor of image b (ascending) pairs with rpn_target_bbox[b, r] (:66-74); positives past
// the T target rows have no partner and are ignored. Optionally writes rpn_pred_box_pos (:64).
__global__ void __launch_bounds__(kLossThreads)
rpn_loss_box_kernel(const int32_t* __restrict__ target, const float4* __restrict__ pred, const float4* __restrict__ target_bbox,
                    int A, int T, RpnLossPart* __restrict__ part, float4* __restrict__ pred_pos, int64_t pred_pos_rows) {
  __shared__ double sd[kLossWarps];
  __shared__ int si[kLossWarps];
  const int b = blockIdx.y, i0 = blockIdx.x * kLossChunk + 4 * threadIdx.x, nchunk = gridDim.x;
  // positives before this chunk: in this image (pairs with the target rows) and in all earlier images (output row)
  int before = 0, earlier = 0;
  for (int64_t c = threadIdx.x; c < (int64_t)b * nchunk + blockIdx.x; c += kLossThreads) {
    const int p = part[c].pos;
    if (c >= (int64_t)b * nchunk) before += p; else earlier += p;
  }
  before = cta_sum(before, si);
  earlier = cta_sum(earlier, si);
  int flags = 0, cnt = 0;
#pragma unroll
  for (int u = 0; u < 4; ++u)
    if (i0 + u < A && target[(int64_t)b * A + i0 + u] == 1) {
      flags |= 1 << u;
      ++cnt;
    }
  // exclusive scan of cnt over the CTA
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int incl = cnt;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  __syncthreads();
  if (lane == 31) si[warp] = incl;
  __syncthreads();
  int off = 0;
  for (int w = 0; w < warp; ++w) off += si[w];
  int r = before + off + incl - cnt;
  double sum = 0.0;
  int used = 0;
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    if (!(flags >> u & 1)) continue;
    const float4 p = __ldg(&pred[(int64_t)b * A + i0 + u]);
    if (pred_pos && (int64_t)earlier + r < pred_pos_rows) pred_pos[(int64_t)earlier + r] = p;
    if (r < T) {
      const float4 t = __ldg(&target_bbox[(int64_t)b * T + r]);
      const float pv[4] = {p.x, p.y, p.z, p.w}, tv[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const float d = fabsf(tv[c] - pv[c]);
        const float less = (d < 1.0f) ? 1.0f : 0.0f;
        sum += (double)((0.5f * less) * (d * d) + (d - 0.5f) * (1.0f - less));   // :79-81
      }
      ++used;
    }
    ++r;
  }
  const double sum_all = cta_sum(sum, sd);
  const int used_all = cta_sum(used, si);
  if (threadIdx.x == 0) {
    part[(int64_t)b * nchunk + blockIdx.x].box_sum = sum_all;
    part[(int64_t)b * nchunk + blockIdx.x].used = used_all;
  }
}

__global__ void __launch_bounds__(kLossThreads)
rpn_loss_final_kernel(const RpnLossPart* __restrict__ part, int64_t n, float* __restrict__ losses, int32_t* __restrict__ num_pos) {
  __shared__ double sd[kLossWarps];
  __shared__ int si[kLossWarps];
  double ce = 0.0, box = 0.0;
  int nz = 0, pos = 0, used = 0;
  for (int64_t c = threadIdx.x; c < n; c += kLossThreads) {
    const RpnLossPart p = part[c];
    ce += p.ce_sum;
    box += p.box_sum;
    nz += p.nz;
    pos += p.pos;
    used += p.used;
  }
  ce = cta_sum(ce, sd);
  box = cta_sum(box, sd);
  nz = cta_sum(nz, si);
  pos = cta_sum(pos, si);
  used = cta_sum(used, si);
  if (threadIdx.x == 0) {
    losses[0] = nz > 0 ? (float)(ce / (double)nz) : 0.0f;                  // K.switch(size > 0, mean, 0) :42
    losses[1] = used > 0 ? (float)(box / (4.0 * (double)used)) : 0.0f;     // :83
    if (num_pos) num_pos[0] = pos;
  }
}

// Both mask-rcnn head losses, one CTA: thread-strided over the B*R ROIs, class loop sequential per ROI.
__global__ void __launch_bounds__(1024)
mrcnn_loss_kernel(const int32_t* __restrict__ target_ids, const float* __restrict__ logits, const float* __restrict__ active,
                  const float4* __restrict__ target_box, const float4* __restrict__ pred_box, int64_t rows, int C,
                  float* __restrict__ losses, float* __restrict__ pred_active_out) {
  __shared__ double sd[32];
  __shared__ int si[32];
  double cls_sum = 0.0, act_sum = 0.0, box_sum = 0.0;
  int box_n = 0;
  const float eps = 1e-7f, hi = 1.0f - 1e-7f;   // K.epsilon()
  for (int64_t r = threadIdx.x; r < rows; r += blockDim.x) {
    const int label = target_ids[r];
    if (logits) {
      const float* x = logits + r * C;
      float m = x[0];
      int arg = 0;
      for (int j = 1; j < C; ++j)
        if (x[j] > m) {   // tf.argmax: first maximum (:113)
          m = x[j];
          arg = j;
        }
      float s = 0.0f;
      for (int j = 0; j < C; ++j) s += f_exp(x[j] - m);
      const float ce = (label >= 0 && label < C) ? f_log(s) - (x[label] - m) : __int_as_float(0x7fc00000);   // :139-142
      const float pa = active[arg];   // batch_active_class_ids[0] gathered at the predicted class (:115)
      if (pred_active_out) pred_active_out[r] = pa;
      cls_sum += (double)(ce * pa);   // :146
      act_sum += (double)pa;
    }
    if (pred_box && label > 0 && label < C) {   // positive ROI (:171): box predicted for its target class (:180-184)
      const float4 t = __ldg(&target_box[r]);
      const float4 p = __ldg(&pred_box[r * C + label]);
      const float tv[4] = {t.x, t.y, t.z, t.w}, pv[4] = {p.x, p.y, p.z, p.w};
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        // K.binary_crossentropy(target, output): clip, logit, sigmoid_cross_entropy_with_logits
        const float o = f_min(f_max(pv[c], eps), hi);
        const float z = f_log(o / (1.0f - o));
        const float l1p = (float)log1p((double)f_exp(-fabsf(z)));
        box_sum += (double)((f_max(z, 0.0f) - z * tv[c]) + l1p);
      }
      ++box_n;
    }
  }
  cls_sum = cta_sum(cls_sum, sd);
  act_sum = cta_sum(act_sum, sd);
  box_sum = cta_sum(box_sum, sd);
  box_n = cta_sum(box_n, si);
  if (threadIdx.x == 0) {
    losses[0] = logits ? (float)(cls_sum / act_sum) : 0.0f;                      // :148 (0/0 = NaN like the reference)
    losses[1] = box_n > 0 ? (float)(box_sum / (4.0 * (double)box_n)) : 0.0f;     // :195-198
  }
}

}  // namespace od

using namespace od;

extern "C" {

size_t od_rpn_loss_workspace_bytes(int64_t batch, int64_t num_anchors) {
  Workspace w(nullptr, 0);
  w.take<RpnLossPart>((size_t)(batch * ((num_anchors + kLossChunk - 1) / kLossChunk) + 1));
  return w.off + 256;
}

int od_rpn_loss_forward(const DLTensor* rpn_target_class, const DLTensor* rpn_class_logits, const DLTensor* rpn_target_bbox,
                        const DLTensor* rpn_pred_box, DLTensor* losses, DLTensor* pred_box_pos, DLTensor* num_pos, void* ws,
                        size_t ws_bytes, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  DeviceScope scope;
  if (rpn_target_class && rpn_target_class->ndim == 3)
    OD_CHECK(check_tensor(rpn_target_class, "rpn_target_class", I32, {kAny, kAny, 1}, 4, scope));
  else
    OD_CHECK(check_tensor(rpn_target_class, "rpn_target_class", I32, {kAny, kAny}, 4, scope));
  const int64_t B = rpn_target_class->shape[0], A = rpn_target_class->shape[1];
  OD_CHECK(check_tensor(rpn_class_logits, "rpn_class_logits", F32, {B, A, 2}, 8, scope));
  OD_CHECK(check_tensor(losses, "losses", F32, {2}, 4, scope));
  const bool with_box = rpn_target_bbox && rpn_pred_box;   // both NULL: class loss only (losses[1] = 0)
  if (!with_box && (rpn_target_bbox || rpn_pred_box || pred_box_pos)) OD_FAIL(OD_ERR_NULL, "rpn_target_bbox and rpn_pred_box go together");
  int64_t T = 0;
  if (with_box) {
    OD_CHECK(check_tensor(rpn_target_bbox, "rpn_target_bbox", F32, {B, kAny, 4}, 16, scope));
    OD_CHECK(check_tensor(rpn_pred_box, "rpn_pred_box", F32, {B, A, 4}, 16, scope));
    T = rpn_target_bbox->shape[1];
  }
  if (A >= (1ll << 31) || B > 65535) OD_FAIL(OD_ERR_PARAM, "supports A < 2^31, B <= 65535");
  OD_CHECK(check_opt_tensor(pred_box_pos, "pred_box_pos", F32, {kAny, 4}, 16, scope));
  const int64_t pos_rows = pred_box_pos ? pred_box_pos->shape[0] : 0;
  OD_CHECK(check_opt_tensor(num_pos, "num_pos", I32, {1}, 4, scope));
  if (!ws) OD_FAIL(OD_ERR_WORKSPACE, "workspace is NULL");
  Workspace w(ws, ws_bytes);
  const int64_t nchunk = (A + kLossChunk - 1) / kLossChunk;
  RpnLossPart* part = w.take<RpnLossPart>((size_t)(B * nchunk + 1));
  if (!w.ok()) OD_FAIL(OD_ERR_WORKSPACE, "workspace %zu < %zu bytes", ws_bytes, w.off);
  if (B > 0 && A > 0) {
    const dim3 grid((unsigned)nchunk, (unsigned)B);
    rpn_loss_class_kernel<<<grid, kLossThreads, 0, st>>>(dptr<int32_t>(rpn_target_class), dptr<float2>(rpn_class_logits), (int)A, part);
    OD_LAUNCH_CHECK("rpn_loss_class_kernel");
    if (with_box) {
      rpn_loss_box_kernel<<<grid, kLossThreads, 0, st>>>(dptr<int32_t>(rpn_target_class), dptr<float4>(rpn_pred_box),
                                                         dptr<float4>(rpn_target_bbox), (int)A, (int)T, part,
                                                         dptr<float4>(pred_box_pos), pos_rows);
      OD_LAUNCH_CHECK("rpn_loss_box_kernel");
    }
  }
  rpn_loss_final_kernel<<<1, kLossThreads, 0, st>>>(part, (B > 0 && A > 0) ? B * nchunk : 0, dptr<float>(losses), dptr<int32_t>(num_pos));
  OD_LAUNCH_CHECK("rpn_loss_final_kernel");
  return OD_OK;
}

int od_mrcnn_loss_forward(const DLTensor* target_class_ids, const DLTensor* pred_logits, const DLTensor* active_class_ids,
                          const DLTensor* target_box, const DLTensor* pred_box, DLTensor* losses, DLTensor* pred_active,
                          void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  DeviceScope scope;
  OD_CHECK(check_tensor(target_class_ids, "mrcnn_target_class_ids", I32, {kAny, kAny}, 4, scope));
  OD_CHECK(check_tensor(losses, "losses", F32, {2}, 4, scope));
  const bool with_cls = pred_logits && active_class_ids, with_box = target_box && pred_box;   // either pair may be NULL
  if ((!with_cls && (pred_logits || active_class_ids || pred_active)) || (!with_box && (target_box || pred_box)) || (!with_cls && !with_box))
    OD_FAIL(OD_ERR_NULL, "pass (mrcnn_pred_logits, batch_active_class_ids) and / or (mrcnn_target_box, mrcnn_pred_box)");
  const int64_t B = target_class_ids->shape[0], R = target_class_ids->shape[1];
  int64_t C = 0;
  if (with_cls) {
    OD_CHECK(check_tensor(pred_logits, "mrcnn_pred_logits", F32, {B, R, kAny}, 4, scope));
    C = pred_logits->shape[2];
    OD_CHECK(check_tensor(active_class_ids, "batch_active_class_ids", F32, {kAny, C}, 4, scope));
    if (active_class_ids->shape[0] < 1) OD_FAIL(OD_ERR_SHAPE, "batch_active_class_ids must be [B,C]");
  }
  if (with_box) {
    OD_CHECK(check_tensor(target_box, "mrcnn_target_box", F32, {B, R, 4}, 16, scope));
    OD_CHECK(check_tensor(pred_box, "mrcnn_pred_box", F32, {B, R, with_cls ? C : kAny, 4}, 16, scope));
    if (!with_cls) C = pred_box->shape[2];
  }
  if (C < 1 || C > (1 << 20)) OD_FAIL(OD_ERR_PARAM, "class count out of range");
  OD_CHECK(check_opt_tensor(pred_active, "pred_active", F32, {B, R}, 4, scope));
  mrcnn_loss_kernel<<<1, 1024, 0, st>>>(dptr<int32_t>(target_class_ids), dptr<float>(pred_logits), dptr<float>(active_class_ids),
                                        dptr<float4>(target_box), dptr<float4>(pred_box), B * R, (int)C, dptr<float>(losses),
                                        dptr<float>(pred_active));
  OD_LAUNCH_CHECK("mrcnn_loss_kernel");
  return OD_OK;
}

}  // extern "C"
