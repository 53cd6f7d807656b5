// proposal.cu — ProposalLayer: top-k -> fused gather/scale/(anchor-gen)/decode/clip -> bitmask NMS -> zero-padded
// proposals. Replaces Proposals.build (proposals_tf.py:136-214), apply_box_deltas (:23-65),
// clip_boxes_to_01 (:67-94) and gen_anchors / gen_anchors_pixel_coord (utils.py:336-369).
#include "anchors.cuh"
#include "nms.cuh"
#include "topk.cuh"

namespace od {

struct ProposalDebugPtrs {
  float* scores;        // [B,K]   (always valid: workspace or debug tensor)
  float4* bbox_delta;   // [B,K] or nullptr
  float4* anchors;      // [B,K] or nullptr
  float4* anchor_delta; // [B,K] or nullptr
  float4* clipped_dbg;  // [B,K] or nullptr
};

// RPN head outputs in their native layout: one [B, n_l, C] block per pyramid level (the reshape of the conv output
// [B,H_l,W_l,a*C], rpn.py:54/66); the reference concatenates them along the anchor axis (training.py:163-166).
struct LevelTable {
  const float* base[OD_MAX_LEVELS];
  int32_t off[OD_MAX_LEVELS + 1];   // first flat anchor index of each level
  int32_t num_levels;
};
template <int C>
__device__ __forceinline__ const float* level_row(const LevelTable& t, int64_t b, int32_t i) {
  int l = 0;
  while (l + 1 < t.num_levels && i >= t.off[l + 1]) ++l;
  const int64_t n_l = t.off[l + 1] - t.off[l];
  return t.base[l] + (b * n_l + (i - t.off[l])) * C;
}

// One thread per selected anchor: 16 B delta + 16 B anchor (or fp64 regeneration) in, 16 B box out.
template <bool LEVELS>
__global__ void __launch_bounds__(256)
proposal_decode_kernel(const float4* __restrict__ bbox, LevelTable lv, const float4* __restrict__ anchors, DevAnchorSpec spec,
                       int use_spec, const int32_t* __restrict__ ix, int64_t total, int K, int A, float4 stddev,
                       float4* __restrict__ clipped, ProposalDebugPtrs dbg) {
  pdl_prologue();
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  const int64_t b = t / K;
  const int32_t i = ix[t];
  const float4 raw = LEVELS ? __ldg(reinterpret_cast<const float4*>(level_row<4>(lv, b, i))) : __ldg(&bbox[b * A + i]);
  const float4 d = make_float4(raw.x * stddev.x, raw.y * stddev.y, raw.z * stddev.z, raw.w * stddev.w);  // :157
  const float4 a = use_spec ? anchor_normalized(spec, i) : __ldg(&anchors[b * A + i]);
  const float4 dec = decode_box(a, d);                                            // :179
  const float4 c = clip_box(dec, make_float4(0.f, 0.f, 1.f, 1.f));                // :183
  clipped[t] = c;
  if (dbg.bbox_delta) dbg.bbox_delta[t] = d;
  if (dbg.anchors) dbg.anchors[t] = a;
  if (dbg.anchor_delta) dbg.anchor_delta[t] = dec;
  if (dbg.clipped_dbg) dbg.clipped_dbg[t] = c;
}

// Foreground probability of every anchor from the per-level class logits: softmax over the (bg, fg) pair
// (rpn.py:58-59, tf.nn.softmax: exp(x - max) / sum) written as one contiguous [B,A] row per image for the top-k.
__global__ void __launch_bounds__(256)
rpn_level_scores_kernel(LevelTable lv, int A, int64_t total, float* __restrict__ scores) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  const int64_t b = t / A;
  const int32_t i = (int32_t)(t - b * A);
  const float2 x = __ldg(reinterpret_cast<const float2*>(level_row<2>(lv, b, i)));
  const float m = (x.x < x.y) ? x.y : x.x;
  const float e0 = f_exp(x.x - m), e1 = f_exp(x.y - m);
  scores[t] = e1 / (e0 + e1);
}

// proposals[b,j] = clipped[b, keep_pos[b,j]] or zeros (tf.pad, :245-246).
__global__ void proposal_gather_kernel(const float4* __restrict__ clipped, const int32_t* __restrict__ keep_pos, int K,
                                       int N, int64_t total, float4* __restrict__ proposals) {
  pdl_prologue();
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  const int64_t b = t / N;
  const int32_t p = keep_pos[t];
  proposals[t] = (p >= 0) ? clipped[b * K + p] : make_float4(0.f, 0.f, 0.f, 0.f);
}

__global__ void apply_box_deltas_kernel(const float4* __restrict__ boxes, const float4* __restrict__ deltas,
                                        int64_t total, float4* __restrict__ out) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < total) out[t] = decode_box(boxes[t], deltas[t]);
}
__global__ void clip_boxes_kernel(const float4* __restrict__ boxes, const float4* __restrict__ window, int per_image,
                                  int64_t K, int64_t total, float4* __restrict__ out) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < total) out[t] = clip_box(boxes[t], window[per_image ? t / K : 0]);
}

__global__ void gen_anchors_norm_kernel(DevAnchorSpec spec, int64_t A, int64_t B, float4* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= A) return;
  const float4 v = anchor_normalized(spec, i);
  for (int64_t b = 0; b < B; ++b) out[b * A + i] = v;
}
__global__ void gen_anchors_pixel_kernel(DevAnchorSpec spec, int64_t A, double* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= A) return;
  double p[4];
  anchor_pixel(spec, i, p);
  for (int c = 0; c < 4; ++c) out[i * 4 + c] = p[c];
}

// utils.norm_boxes (utils.py:181-196: fp64 divide, cast to fp32) and utils.norm_boxes_tf (utils.py:198-210: fp32
// throughout, scale = float32(h) - 1.0f). One thread per box.
template <typename TIn, bool TF32>
__global__ void norm_boxes_kernel(const TIn* __restrict__ in, int64_t n, int32_t image_h, int32_t image_w,
                                  float4* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const TIn* p = in + 4 * i;
  float4 r;
  if (TF32) {
    const float sh = __fsub_rn((float)image_h, 1.0f), sw = __fsub_rn((float)image_w, 1.0f);
    r.x = __fdiv_rn(__fsub_rn((float)p[0], 0.0f), sh);
    r.y = __fdiv_rn(__fsub_rn((float)p[1], 0.0f), sw);
    r.z = __fdiv_rn(__fsub_rn((float)p[2], 1.0f), sh);
    r.w = __fdiv_rn(__fsub_rn((float)p[3], 1.0f), sw);
  } else {
    const double sh = (double)(image_h - 1), sw = (double)(image_w - 1);
    r.x = (float)(((double)p[0] - 0.0) / sh);
    r.y = (float)(((double)p[1] - 0.0) / sw);
    r.z = (float)(((double)p[2] - 1.0) / sh);
    r.w = (float)(((double)p[3] - 1.0) / sw);
  }
  out[i] = r;
}

struct ProposalWs {
  int32_t* ix;
  float* scores;
  float4* clipped;
  int32_t* keep_pos;
  int32_t* num_kept;
  void* topk_ws;
  size_t topk_bytes;
  void* nms_ws;
  size_t nms_bytes;
};
static size_t carve_proposal_ws(Workspace& w, int64_t B, int64_t A, int64_t K, int64_t N, ProposalWs* out) {
  ProposalWs p;
  p.ix = w.take<int32_t>((size_t)(B * K));
  p.scores = w.take<float>((size_t)(B * K));
  p.clipped = w.take<float4>((size_t)(B * K));
  p.keep_pos = w.take<int32_t>((size_t)(B * N));
  p.num_kept = w.take<int32_t>((size_t)B);
  p.topk_bytes = topk_workspace_bytes(B, A, K);
  p.topk_ws = w.take<char>(p.topk_bytes);
  p.nms_bytes = nms_sorted_workspace_bytes(B, K);
  p.nms_ws = w.take<char>(p.nms_bytes);
  if (out) *out = p;
  return w.off + 256;
}

}  // namespace od

using namespace od;

extern "C" {

int64_t od_anchor_count(const od_anchor_spec* spec) {
  DevAnchorSpec d;
  if (make_dev_anchor_spec(spec, &d) != OD_OK) return -1;
  return d.offset[d.num_levels];
}

int od_gen_anchors(const od_anchor_spec* spec, int normalized, DLTensor* anchors, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  DevAnchorSpec d;
  OD_CHECK(make_dev_anchor_spec(spec, &d));
  const int64_t A = d.offset[d.num_levels];
  DeviceScope scope;
  if (normalized) {
    OD_CHECK(check_tensor(anchors, "anchors", F32, {kAny, A, 4}, 16, scope));
    if (A == 0 || anchors->shape[0] == 0) return OD_OK;
    gen_anchors_norm_kernel<<<(unsigned)((A + 255) / 256), 256, 0, st>>>(d, A, anchors->shape[0], dptr<float4>(anchors));
  } else {
    OD_CHECK(check_tensor(anchors, "anchors", F64, {A, 4}, 8, scope));
    if (A == 0) return OD_OK;
    gen_anchors_pixel_kernel<<<(unsigned)((A + 255) / 256), 256, 0, st>>>(d, A, dptr<double>(anchors));
  }
  OD_LAUNCH_CHECK("gen_anchors");
  return OD_OK;
}

int od_apply_box_deltas(const DLTensor* boxes, const DLTensor* deltas, DLTensor* out, void* stream) {
  DeviceScope scope;
  OD_CHECK(check_tensor(boxes, "boxes", F32, {kAny, kAny, 4}, 16, scope));
  OD_CHECK(check_tensor(deltas, "deltas", F32, {boxes->shape[0], boxes->shape[1], 4}, 16, scope));
  OD_CHECK(check_tensor(out, "out", F32, {boxes->shape[0], boxes->shape[1], 4}, 16, scope));
  const int64_t total = boxes->shape[0] * boxes->shape[1];
  if (total == 0) return OD_OK;
  apply_box_deltas_kernel<<<(unsigned)((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      dptr<float4>(boxes), dptr<float4>(deltas), total, dptr<float4>(out));
  OD_LAUNCH_CHECK("apply_box_deltas_kernel");
  return OD_OK;
}

int od_clip_boxes(const DLTensor* boxes, const DLTensor* window, DLTensor* out, void* stream) {
  DeviceScope scope;
  OD_CHECK(check_tensor(boxes, "boxes", F32, {kAny, kAny, 4}, 16, scope));
  const int per_image = window && window->ndim == 2;   // window [B,4], else [4]
  if (per_image) OD_CHECK(check_tensor(window, "window", F32, {boxes->shape[0], 4}, 16, scope));
  else OD_CHECK(check_tensor(window, "window", F32, {4}, 16, scope));
  OD_CHECK(check_tensor(out, "out", F32, {boxes->shape[0], boxes->shape[1], 4}, 16, scope));
  const int64_t total = boxes->shape[0] * boxes->shape[1];
  if (total == 0) return OD_OK;
  clip_boxes_kernel<<<(unsigned)((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      dptr<float4>(boxes), dptr<float4>(window), per_image, boxes->shape[1], total, dptr<float4>(out));
  OD_LAUNCH_CHECK("clip_boxes_kernel");
  return OD_OK;
}

int od_norm_boxes(const DLTensor* boxes, int32_t image_h, int32_t image_w, int32_t tf_float32, DLTensor* out, void* stream) {
  DeviceScope scope;
  if (!boxes) OD_FAIL(OD_ERR_NULL, "boxes is NULL");
  const bool is_i32 = boxes->dtype.code == kDLInt && boxes->dtype.bits == 32;
  const bool is_f64 = boxes->dtype.code == kDLFloat && boxes->dtype.bits == 64;
  OD_CHECK(check_tensor(boxes, "boxes", is_i32 ? I32 : (is_f64 ? F64 : F32), nullptr, -1, is_f64 ? 8 : 4, scope));
  if (boxes->ndim < 1) OD_FAIL(OD_ERR_SHAPE, "boxes must be [...,4]");
  if (boxes->shape[boxes->ndim - 1] != 4)
    OD_FAIL(OD_ERR_SHAPE, "boxes: extent %d is %lld, expected 4", boxes->ndim - 1, (long long)boxes->shape[boxes->ndim - 1]);
  OD_CHECK(check_tensor(out, "out", F32, boxes->shape, boxes->ndim, 16, scope));
  if (tf_float32 && !(!is_i32 && !is_f64)) OD_FAIL(OD_ERR_DTYPE, "norm_boxes_tf takes float32 boxes");
  const int64_t n = numel(boxes) / 4;
  if (n == 0) return OD_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const unsigned grid = (unsigned)((n + 127) / 128);
  if (tf_float32) norm_boxes_kernel<float, true><<<grid, 128, 0, st>>>(dptr<float>(boxes), n, image_h, image_w, dptr<float4>(out));
  else if (is_i32) norm_boxes_kernel<int32_t, false><<<grid, 128, 0, st>>>(dptr<int32_t>(boxes), n, image_h, image_w, dptr<float4>(out));
  else if (is_f64) norm_boxes_kernel<double, false><<<grid, 128, 0, st>>>(dptr<double>(boxes), n, image_h, image_w, dptr<float4>(out));
  else norm_boxes_kernel<float, false><<<grid, 128, 0, st>>>(dptr<float>(boxes), n, image_h, image_w, dptr<float4>(out));
  OD_LAUNCH_CHECK("norm_boxes_kernel");
  return OD_OK;
}

size_t od_proposal_workspace_bytes(int64_t batch, int64_t num_anchors, const od_proposal_params* p) {
  if (!p) return 0;
  const int64_t K = p->pre_nms_limit < num_anchors ? p->pre_nms_limit : num_anchors;
  Workspace w(nullptr, 0);
  return carve_proposal_ws(w, batch, num_anchors, K, p->post_nms_count, nullptr);
}

}  // extern "C"

namespace od {
// Shared body of od_proposal_forward / od_proposal_forward_levels. `scores` addresses the fg score of anchor i of image b at
// scores[b * score_sb + i * score_sa]; with `logits` (the per-level class logits), it is a workspace row that is first
// filled from them. The deltas come from `rpn_bbox4` ([B,A,4]) or, when it is NULL, from `lv`. `p` is the carved
// workspace. Shapes B, A are those of the caller's (virtual) [B,A,.] tensors.
static int proposal_core(float* scores_src, int64_t score_sb, int64_t score_sa, const LevelTable* logits, const float4* rpn_bbox4,
                         const LevelTable& lv, int64_t B, int64_t A, const DLTensor* anchors, const od_anchor_spec* spec,
                         const od_proposal_params* params, DLTensor* proposals, const od_proposal_debug* debug, ProposalWs& p,
                         DeviceScope& scope, cudaStream_t st) {
  const int64_t K = params->pre_nms_limit < A ? params->pre_nms_limit : A;
  const int64_t N = params->post_nms_count;
  OD_CHECK(check_tensor(proposals, "proposals", F32, {B, N, 4}, 16, scope));
  DevAnchorSpec dspec;
  memset(&dspec, 0, sizeof(dspec));
  int use_spec = 0;
  if (anchors) {
    OD_CHECK(check_tensor(anchors, "anchors", F32, {B, A, 4}, 16, scope));
  } else {
    if (!spec) OD_FAIL(OD_ERR_NULL, "either anchors or an anchor spec is required");
    OD_CHECK(make_dev_anchor_spec(spec, &dspec));
    if (dspec.offset[dspec.num_levels] != A) OD_FAIL(OD_ERR_SHAPE, "anchor spec yields %lld anchors, inputs have %lld", (long long)dspec.offset[dspec.num_levels], (long long)A);
    use_spec = 1;
  }
  od_proposal_debug dbg;
  memset(&dbg, 0, sizeof(dbg));
  if (debug) dbg = *debug;
  OD_CHECK(check_opt_tensor(dbg.ix, "debug.ix", I32, {B, K}, 4, scope));
  OD_CHECK(check_opt_tensor(dbg.scores, "debug.scores", F32, {B, K}, 4, scope));
  OD_CHECK(check_opt_tensor(dbg.bbox_delta, "debug.bbox_delta", F32, {B, K, 4}, 16, scope));
  OD_CHECK(check_opt_tensor(dbg.anchors, "debug.anchors", F32, {B, K, 4}, 16, scope));
  OD_CHECK(check_opt_tensor(dbg.anchor_delta, "debug.anchor_delta", F32, {B, K, 4}, 16, scope));
  OD_CHECK(check_opt_tensor(dbg.anchor_delta_clipped, "debug.anchor_delta_clipped", F32, {B, K, 4}, 16, scope));
  OD_CHECK(check_opt_tensor(dbg.keep_idx, "debug.keep_idx", I32, {B, N}, 4, scope));
  OD_CHECK(check_opt_tensor(dbg.num_kept, "debug.num_kept", I32, {B}, 4, scope));
  if (B == 0 || N == 0) return OD_OK;
  if (logits && B * A > 0) {
    rpn_level_scores_kernel<<<(unsigned)((B * A + 255) / 256), 256, 0, st>>>(*logits, (int)A, B * A, scores_src);
    OD_LAUNCH_CHECK("rpn_level_scores_kernel");
  }
  int32_t* ix = dbg.ix ? dptr<int32_t>(dbg.ix) : p.ix;
  float* scores = dbg.scores ? dptr<float>(dbg.scores) : nullptr;  // only materialised on request
  int32_t* keep_pos = dbg.keep_idx ? dptr<int32_t>(dbg.keep_idx) : p.keep_pos;
  int32_t* num_kept = dbg.num_kept ? dptr<int32_t>(dbg.num_kept) : p.num_kept;

  // scores = probs[:,:,1]  (:153) -> top-k (:169)
  OD_CHECK(topk_launch(scores_src, B, A, score_sb, score_sa, K, ix, scores, p.topk_ws, p.topk_bytes, st));
  if (K > 0) {
    ProposalDebugPtrs dp;
    dp.scores = scores;
    dp.bbox_delta = dptr<float4>(dbg.bbox_delta);
    dp.anchors = dptr<float4>(dbg.anchors);
    dp.anchor_delta = dptr<float4>(dbg.anchor_delta);
    dp.clipped_dbg = dptr<float4>(dbg.anchor_delta_clipped);
    const int64_t total = B * K;
    const float4 sd = make_float4(params->bbox_stddev[0], params->bbox_stddev[1], params->bbox_stddev[2], params->bbox_stddev[3]);
    if (rpn_bbox4)
      OD_CUDA(launch_pdl(proposal_decode_kernel<false>, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, st,
          rpn_bbox4, lv, dptr<float4>(anchors), dspec, use_spec, ix, total, (int)K, (int)A, sd, p.clipped, dp));
    else
      OD_CUDA(launch_pdl(proposal_decode_kernel<true>, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, st,
          (const float4*)nullptr, lv, dptr<float4>(anchors), dspec, use_spec, ix, total, (int)K, (int)A, sd, p.clipped, dp));
    OD_LAUNCH_CHECK("proposal_decode_kernel");
  }
  // per-image NMS over boxes already in (score desc, index asc) order (:188-196, :234)
  OD_CHECK(nms_sorted_launch(p.clipped, nullptr, nullptr, B, K, params->nms_threshold, N, keep_pos, num_kept, nullptr,
                             p.nms_ws, p.nms_bytes, st));
  const int64_t total = B * N;
  OD_CUDA(launch_pdl(proposal_gather_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, st, p.clipped, keep_pos, (int)K, (int)N, total,
                                                                         dptr<float4>(proposals)));
  OD_LAUNCH_CHECK("proposal_gather_kernel");
  return OD_OK;
}
}  // namespace od

extern "C" {

int od_proposal_forward(const DLTensor* rpn_class_probs, const DLTensor* rpn_bbox, const DLTensor* anchors,
                        const od_anchor_spec* spec, const od_proposal_params* params, DLTensor* proposals,
                        const od_proposal_debug* debug, void* ws, size_t ws_bytes, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (!params) OD_FAIL(OD_ERR_NULL, "params is NULL");
  DeviceScope scope;
  OD_CHECK(check_tensor(rpn_class_probs, "rpn_class_probs", F32, {kAny, kAny, 2}, 4, scope));
  const int64_t B = rpn_class_probs->shape[0], A = rpn_class_probs->shape[1];
  OD_CHECK(check_tensor(rpn_bbox, "rpn_bbox", F32, {B, A, 4}, 16, scope));
  if (params->pre_nms_limit < 0 || params->post_nms_count < 0) OD_FAIL(OD_ERR_PARAM, "negative counts");
  const int64_t K = params->pre_nms_limit < A ? params->pre_nms_limit : A;
  const int64_t N = params->post_nms_count;
  ProposalWs p;
  memset(&p, 0, sizeof(p));
  if (B != 0 && N != 0) {
    if (!ws) OD_FAIL(OD_ERR_WORKSPACE, "workspace is NULL");
    Workspace w(ws, ws_bytes);
    carve_proposal_ws(w, B, A, K, N, &p);
    if (!w.ok()) OD_FAIL(OD_ERR_WORKSPACE, "workspace %zu < %zu bytes", ws_bytes, w.off);
  }
  LevelTable lv;
  memset(&lv, 0, sizeof(lv));
  // scores = probs[:,:,1]  (:153)
  return proposal_core(dptr<float>(rpn_class_probs) + 1, 2 * A, 2, nullptr, dptr<float4>(rpn_bbox), lv, B, A, anchors, spec,
                       params, proposals, debug, p, scope, st);
}

size_t od_proposal_levels_workspace_bytes(int64_t batch, int64_t num_anchors, const od_proposal_params* p) {
  if (!p) return 0;
  const int64_t K = p->pre_nms_limit < num_anchors ? p->pre_nms_limit : num_anchors;
  Workspace w(nullptr, 0);
  w.take<float>((size_t)(batch * num_anchors));
  return carve_proposal_ws(w, batch, num_anchors, K, p->post_nms_count, nullptr);
}

int od_proposal_forward_levels(const DLTensor* const* class_logits, const DLTensor* const* bbox, int32_t num_levels,
                               const DLTensor* anchors, const od_anchor_spec* spec, const od_proposal_params* params,
                               DLTensor* proposals, const od_proposal_debug* debug, void* ws, size_t ws_bytes, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (!params || !class_logits || !bbox) OD_FAIL(OD_ERR_NULL, "params / class_logits / bbox is NULL");
  if (num_levels < 1 || num_levels > OD_MAX_LEVELS) OD_FAIL(OD_ERR_PARAM, "num_levels %d out of range", num_levels);
  if (params->pre_nms_limit < 0 || params->post_nms_count < 0) OD_FAIL(OD_ERR_PARAM, "negative counts");
  DeviceScope scope;
  LevelTable lc, lb;
  memset(&lc, 0, sizeof(lc));
  memset(&lb, 0, sizeof(lb));
  lc.num_levels = lb.num_levels = num_levels;
  int64_t B = kAny, A = 0;   // B: that of the first level
  for (int l = 0; l < num_levels; ++l) {
    const DLTensor* c = class_logits[l];
    const DLTensor* d = bbox[l];
    OD_CHECK(check_tensor(c, "class_logits[l]", F32, {B, kAny, kAny, kAny}, 8, scope));
    B = c->shape[0];
    if (c->shape[3] % 2) OD_FAIL(OD_ERR_SHAPE, "class_logits[l]: extent 3 is %lld, expected an even value (level %d)", (long long)c->shape[3], l);
    OD_CHECK(check_tensor(d, "bbox[l]", F32, {B, c->shape[1], c->shape[2], 2 * c->shape[3]}, 16, scope));
    const int64_t n_l = c->shape[1] * c->shape[2] * (c->shape[3] / 2);
    lc.base[l] = dptr<float>(c);
    lb.base[l] = dptr<float>(d);
    lc.off[l] = lb.off[l] = (int32_t)A;
    A += n_l;
    if (A >= (1ll << 31)) OD_FAIL(OD_ERR_PARAM, "too many anchors");
  }
  for (int l = num_levels; l <= OD_MAX_LEVELS; ++l) lc.off[l] = lb.off[l] = (int32_t)A;
  const int64_t K = params->pre_nms_limit < A ? params->pre_nms_limit : A;
  const int64_t N = params->post_nms_count;
  ProposalWs p;
  memset(&p, 0, sizeof(p));
  float* scores = nullptr;
  if (B != 0 && N != 0) {
    if (!ws) OD_FAIL(OD_ERR_WORKSPACE, "workspace is NULL");
    Workspace w(ws, ws_bytes);
    scores = w.take<float>((size_t)(B * A));
    carve_proposal_ws(w, B, A, K, N, &p);
    if (!w.ok()) OD_FAIL(OD_ERR_WORKSPACE, "workspace %zu < %zu bytes", ws_bytes, w.off);
  }
  return proposal_core(scores, A, 1, &lc, nullptr, lb, B, A, anchors, spec, params, proposals, debug, p, scope, st);
}

}  // extern "C"
