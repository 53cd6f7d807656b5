/*
 * odhead_oracle.c — CPU ORACLE. TEST INFRASTRUCTURE ONLY.
 *
 * A plain-C restatement of the reference's detection-head algorithm
 * (Sardhendu/ObjectDetection). Only tests/, __graft_entry__.smoke() and
 * bench.py's cpu_baseline / --impl reference legs may load this library; the
 * product (objectdetection_b200 + libodhead.so) never does.
 *
 * PARITY STATUS
 *   pinned   : anchor generation, norm/denorm boxes, stage shapes, numpy IoU/NMS,
 *              FasterRCNN numpy decode/clip/filter/NMS — checked against golden
 *              vectors produced by importing the reference's own numpy functions
 *              (tests/golden/make_golden.py) and against the notebook constants
 *              G1–G8 of SURVEY.md §4.
 *   anchored : the three TensorFlow kernels the layers call (tf.nn.top_k,
 *              tf.image.non_max_suppression, tf.image.crop_and_resize).
 *              TensorFlow (1.8–1.10, un-pinned and un-vendored by the
 *              reference) is a third-party dependency absent from the tree and
 *              not installable here, so these are restated from the published
 *              CPU kernels core/kernels/{topk_op,non_max_suppression_op,
 *              crop_and_resize_op}.cc and checked against the known-answer
 *              vectors of TensorFlow's own kernel tests
 *              (crop_and_resize_op_test.cc, non_max_suppression_op_test.cc;
 *              restated in tests/test_tf_known_answers.py — not produced by
 *              running TensorFlow) and against independent implementations
 *              (torchvision NMS, torch grid_sample).
 *   UNPINNED : the four layers composed from those kernels (ProposalLayer,
 *              PyramidROIAlign, DetectionTargetLayer, DetectionLayer) and the
 *              mask targets: the reference ships no recorded outputs for them
 *              and cannot be run here: "parity unpinned". The restatement
 *              follows the reference's graph code line by line (cited per
 *              function).
 *
 * Numeric conventions (shared with the CUDA kernels so integer outputs are
 * bit-exact): fp32 arithmetic in the reference's operation order, no FMA
 * contraction (build with -ffp-contract=off), IEEE division/sqrt; exp/log are
 * the correctly-rounded fp32 values obtained by evaluating in fp64 and rounding;
 * min/max are the `(b<a)?b:a` / `(a<b)?b:a` forms of std::min/std::max (NaN
 * propagates from the first operand); ties order by lower index.
 *
 * Build: see oracle/Makefile  (gcc -O2 -ffp-contract=off -fopenmp -shared -fPIC).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <limits.h>

#define ORC_API __attribute__((visibility("default")))

static inline float f_min(float a, float b) { return (b < a) ? b : a; }
static inline float f_max(float a, float b) { return (a < b) ? b : a; }
static inline float f_exp(float x) { return (float)exp((double)x); }
static inline float f_log(float x) { return (float)log((double)x); }

/* float -> int32 with x86 cvttss2si behaviour (NaN / out of range -> INT_MIN). */
static inline int32_t f_to_i32(float r) {
  if (!(r > -2147483904.0f && r < 2147483648.0f)) return INT32_MIN;
  return (int32_t)r;
}
static inline int32_t i32_add_wrap(int32_t a, int32_t b) {
  return (int32_t)((uint32_t)a + (uint32_t)b);
}

/* Order-preserving map float -> uint32 (larger float = larger key); -0 == +0. Every NaN, of either sign and any
 * payload, is one value above +inf (numpy's sort order; TF's comparator leaves NaNs unordered), so NaN ties go to
 * the lower index like any other tie. */
static inline uint32_t score_key(float s) {
  uint32_t b;
  if (s != s) return 0xFFFFFFFFu;
  s = s + 0.0f;
  memcpy(&b, &s, 4);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
/* (score desc, index asc) == composite desc */
static inline uint64_t composite_key(float s, uint32_t idx) {
  return ((uint64_t)score_key(s) << 32) | (uint64_t)(0xFFFFFFFFu - idx);
}
static inline uint32_t composite_index(uint64_t c) { return 0xFFFFFFFFu - (uint32_t)(c & 0xFFFFFFFFu); }

static int cmp_u64_desc(const void* a, const void* b) {
  uint64_t x = *(const uint64_t*)a, y = *(const uint64_t*)b;
  return (x < y) - (x > y);
}

/* Partition so that the k largest of v[0..n) occupy v[0..k) (unordered). */
static void select_k_largest(uint64_t* v, int64_t n, int64_t k) {
  int64_t lo = 0, hi = n - 1;
  if (k <= 0 || k >= n) return;
  while (lo < hi) {
    int64_t mid = lo + (hi - lo) / 2;
    uint64_t a = v[lo], b = v[mid], c = v[hi], pivot;
    pivot = (a > b) ? ((b > c) ? b : ((a > c) ? c : a)) : ((a > c) ? a : ((b > c) ? c : b));
    int64_t i = lo, j = hi;
    while (i <= j) {
      while (v[i] > pivot) i++;
      while (v[j] < pivot) j--;
      if (i <= j) { uint64_t t = v[i]; v[i] = v[j]; v[j] = t; i++; j--; }
    }
    if (k - 1 <= j) hi = j;
    else if (k - 1 >= i) lo = i;
    else break;
  }
}

/* ------------------------------------------------------------------------- */
/* tf.nn.top_k(sorted=True): k largest per row, descending, ties -> lower index.
 * Call sites: proposals_tf.py:169, maskrcnn.py:171, detection.py:221.          */
ORC_API void orc_topk(const float* scores, int64_t rows, int64_t cols, int64_t row_stride,
                      int64_t col_stride, int64_t k, int32_t* idx_out, float* val_out) {
#pragma omp parallel for schedule(dynamic, 1)
  for (int64_t r = 0; r < rows; ++r) {
    const float* s = scores + r * row_stride;
    uint64_t* keys = (uint64_t*)malloc(sizeof(uint64_t) * (size_t)(cols > 0 ? cols : 1));
    for (int64_t i = 0; i < cols; ++i) keys[i] = composite_key(s[i * col_stride], (uint32_t)i);
    select_k_largest(keys, cols, k);
    qsort(keys, (size_t)k, sizeof(uint64_t), cmp_u64_desc);
    for (int64_t i = 0; i < k; ++i) {
      uint32_t ix = composite_index(keys[i]);
      idx_out[r * k + i] = (int32_t)ix;
      if (val_out) val_out[r * k + i] = s[(int64_t)ix * col_stride];
    }
    free(keys);
  }
}

/* ------------------------------------------------------------------------- */
/* apply_box_deltas, proposals_tf.py:46-61 (fp32, reference op order).          */
static inline void decode_one(const float* a, const float* d, float* o) {
  float height = a[2] - a[0];
  float width = a[3] - a[1];
  float center_y = a[0] + 0.5f * height;
  float center_x = a[1] + 0.5f * width;
  center_y = center_y + d[0] * height;
  center_x = center_x + d[1] * width;
  height = height * f_exp(d[2]);
  width = width * f_exp(d[3]);
  float y1 = center_y - 0.5f * height;
  float x1 = center_x - 0.5f * width;
  float y2 = y1 + height;
  float x2 = x1 + width;
  o[0] = y1; o[1] = x1; o[2] = y2; o[3] = x2;
}
ORC_API void orc_apply_box_deltas(const float* boxes, const float* deltas, int64_t n, float* out) {
  for (int64_t i = 0; i < n; ++i) decode_one(boxes + 4 * i, deltas + 4 * i, out + 4 * i);
}
/* clip_boxes_to_01, proposals_tf.py:86-94: max(min(v, hi), lo). window = (wy1,wx1,wy2,wx2). */
static inline void clip_one(const float* b, const float* w, float* o) {
  o[0] = f_max(f_min(b[0], w[2]), w[0]);
  o[1] = f_max(f_min(b[1], w[3]), w[1]);
  o[2] = f_max(f_min(b[2], w[2]), w[0]);
  o[3] = f_max(f_min(b[3], w[3]), w[1]);
}
ORC_API void orc_clip_boxes(const float* boxes, const float* window, int64_t n, float* out) {
  for (int64_t i = 0; i < n; ++i) clip_one(boxes + 4 * i, window, out + 4 * i);
}

/* ------------------------------------------------------------------------- */
/* tf.image.non_max_suppression (V2): TF core/kernels/non_max_suppression_op.cc.
 * IoU with corner canonicalisation and area<=0 -> 0; suppress iff IoU > thr.   */
static inline float tf_iou(const float* bi, const float* bj) {
  const float ymin_i = f_min(bi[0], bi[2]), xmin_i = f_min(bi[1], bi[3]);
  const float ymax_i = f_max(bi[0], bi[2]), xmax_i = f_max(bi[1], bi[3]);
  const float ymin_j = f_min(bj[0], bj[2]), xmin_j = f_min(bj[1], bj[3]);
  const float ymax_j = f_max(bj[0], bj[2]), xmax_j = f_max(bj[1], bj[3]);
  const float area_i = (ymax_i - ymin_i) * (xmax_i - xmin_i);
  const float area_j = (ymax_j - ymin_j) * (xmax_j - xmin_j);
  if (area_i <= 0 || area_j <= 0) return 0.0f;
  const float iymin = f_max(ymin_i, ymin_j), ixmin = f_max(xmin_i, xmin_j);
  const float iymax = f_min(ymax_i, ymax_j), ixmax = f_min(xmax_i, xmax_j);
  const float inter = f_max(iymax - iymin, 0.0f) * f_max(ixmax - ixmin, 0.0f);
  return inter / (area_i + area_j - inter);
}
ORC_API float orc_tf_iou(const float* bi, const float* bj) { return tf_iou(bi, bj); }

/* Returns the number kept; keep[] holds box indices in selection order. */
ORC_API int32_t orc_nms(const float* boxes, const float* scores, int32_t n, int32_t max_out,
                        float thr, int32_t* keep) {
  if (n <= 0 || max_out <= 0) return 0;
  uint64_t* order = (uint64_t*)malloc(sizeof(uint64_t) * (size_t)n);
  for (int32_t i = 0; i < n; ++i) order[i] = composite_key(scores[i], (uint32_t)i);
  qsort(order, (size_t)n, sizeof(uint64_t), cmp_u64_desc);
  int32_t cnt = 0;
  for (int32_t c = 0; c < n && cnt < max_out; ++c) {
    const int32_t i = (int32_t)composite_index(order[c]);
    int ok = 1;
    for (int32_t j = cnt - 1; j >= 0; --j) {
      if (tf_iou(boxes + 4 * (int64_t)i, boxes + 4 * (int64_t)keep[j]) > thr) { ok = 0; break; }
    }
    if (ok) keep[cnt++] = i;
  }
  free(order);
  return cnt;
}

/* ------------------------------------------------------------------------- */
/* tf.image.crop_and_resize(method="bilinear"): TF core/kernels/crop_and_resize_op.cc
 * image [B,H,W,D] NHWC, boxes [n,4], box_ind [n] -> out [n,ch,cw,D].
 * Call sites: maskrcnn.py:152, FasterRCNN/building_blocks/fastrcnn.py:68.        */
ORC_API void orc_crop_and_resize(const float* image, int32_t B, int32_t H, int32_t W, int32_t D,
                                 const float* boxes, const int32_t* box_ind, int32_t n,
                                 int32_t ch, int32_t cw, float extrapolation, float* out) {
#pragma omp parallel for schedule(dynamic, 4)
  for (int32_t b = 0; b < n; ++b) {
    const float y1 = boxes[4 * b + 0], x1 = boxes[4 * b + 1];
    const float y2 = boxes[4 * b + 2], x2 = boxes[4 * b + 3];
    const int32_t b_in = box_ind[b];
    if (b_in < 0 || b_in >= B) continue;
    const float* img = image + (int64_t)b_in * H * W * D;
    float* o = out + (int64_t)b * ch * cw * D;
    const float height_scale = (ch > 1) ? (y2 - y1) * (float)(H - 1) / (float)(ch - 1) : 0.0f;
    const float width_scale = (cw > 1) ? (x2 - x1) * (float)(W - 1) / (float)(cw - 1) : 0.0f;
    for (int32_t y = 0; y < ch; ++y) {
      const float in_y = (ch > 1) ? y1 * (float)(H - 1) + (float)y * height_scale
                                  : (float)(0.5 * (double)(y1 + y2) * (double)(H - 1));
      float* orow = o + (int64_t)y * cw * D;
      if (!(in_y >= 0) || !(in_y <= (float)(H - 1))) {   /* NaN treated as out of range */
        for (int64_t t = 0; t < (int64_t)cw * D; ++t) orow[t] = extrapolation;
        continue;
      }
      const int32_t top = (int32_t)floorf(in_y), bot = (int32_t)ceilf(in_y);
      const float y_lerp = in_y - (float)top;
      for (int32_t x = 0; x < cw; ++x) {
        const float in_x = (cw > 1) ? x1 * (float)(W - 1) + (float)x * width_scale
                                    : (float)(0.5 * (double)(x1 + x2) * (double)(W - 1));
        float* op = orow + (int64_t)x * D;
        if (!(in_x >= 0) || !(in_x <= (float)(W - 1))) {
          for (int32_t d = 0; d < D; ++d) op[d] = extrapolation;
          continue;
        }
        const int32_t left = (int32_t)floorf(in_x), right = (int32_t)ceilf(in_x);
        const float x_lerp = in_x - (float)left;
        const float* tl = img + ((int64_t)top * W + left) * D;
        const float* tr = img + ((int64_t)top * W + right) * D;
        const float* bl = img + ((int64_t)bot * W + left) * D;
        const float* br = img + ((int64_t)bot * W + right) * D;
        for (int32_t d = 0; d < D; ++d) {
          const float t = tl[d] + (tr[d] - tl[d]) * x_lerp;
          const float bo = bl[d] + (br[d] - bl[d]) * x_lerp;
          op[d] = t + (bo - t) * y_lerp;
        }
      }
    }
  }
}

/* FPN level assignment, maskrcnn.py:104-122. */
ORC_API int32_t orc_roi_level(const float* roi, int32_t image_h, int32_t image_w,
                              int32_t min_level, int32_t max_level) {
  const float h = roi[2] - roi[0];
  const float w = roi[3] - roi[1];
  const float image_area = (float)(image_h * image_w);
  const float denom = 224.0f / sqrtf(image_area);
  const float v = sqrtf(h * w) / denom;
  const float lv = f_log(v) / f_log(2.0f);
  const float r = nearbyintf(lv);                 /* tf.round = half to even */
  int32_t level = i32_add_wrap(4, f_to_i32(r));
  level = (level > min_level) ? level : min_level;  /* tf.maximum(min_k, .) */
  level = (level < max_level) ? level : max_level;  /* tf.minimum(max_k, .) */
  return level;
}

/* MaskRCNN.roi_pooling, maskrcnn.py:74-187. fmaps[l] is level (min_level + l).
 * out [B*N, ph, pw, D], row b*N+n <-> rois[b,n]; levels_out [B*N] may be NULL. */
ORC_API void orc_pyramid_roi_align(const float* const* fmaps, const int32_t* fh, const int32_t* fw,
                                   int32_t num_levels, int32_t min_level, int32_t B, int32_t D,
                                   const float* rois, int32_t N, int32_t image_h, int32_t image_w,
                                   int32_t ph, int32_t pw, float* out, int32_t* levels_out) {
  const int32_t max_level = min_level + num_levels - 1;
  const int64_t total = (int64_t)B * N;
  int32_t* lv = (int32_t*)malloc(sizeof(int32_t) * (size_t)(total > 0 ? total : 1));
  int32_t* bi = (int32_t*)malloc(sizeof(int32_t) * (size_t)(total > 0 ? total : 1));
  for (int64_t i = 0; i < total; ++i) {
    lv[i] = orc_roi_level(rois + 4 * i, image_h, image_w, min_level, max_level);
    if (levels_out) levels_out[i] = lv[i];
  }
  for (int32_t l = 0; l < num_levels; ++l) {
    /* box_ind < 0 skips the crop: rows of other levels are left to their own pass. */
    for (int64_t i = 0; i < total; ++i) bi[i] = (lv[i] == min_level + l) ? (int32_t)(i / N) : -1;
    orc_crop_and_resize(fmaps[l], B, fh[l], fw[l], D, rois, bi, (int32_t)total, ph, pw, 0.0f, out);
  }
  free(lv);
  free(bi);
}

/* ------------------------------------------------------------------------- */
/* Proposals.build, proposals_tf.py:136-214. One image per OpenMP task.
 * Optional outputs may be NULL. keep_out is [B,N] padded with -1.            */
ORC_API void orc_proposal_forward(const float* probs /*[B,A,2]*/, const float* bbox /*[B,A,4]*/,
                                  const float* anchors /*[B,A,4]*/, int32_t B, int32_t A,
                                  const float* stddev /*[4]*/, int32_t pre_nms_limit, int32_t N,
                                  float nms_thr, float* proposals /*[B,N,4]*/,
                                  int32_t* ix_out /*[B,K]*/, float* scores_out /*[B,K]*/,
                                  float* delta_out /*[B,K,4]*/, float* anchors_out /*[B,K,4]*/,
                                  float* decoded_out /*[B,K,4]*/, float* clipped_out /*[B,K,4]*/,
                                  int32_t* keep_out /*[B,N]*/, int32_t* num_kept_out /*[B]*/) {
  const int32_t K = (pre_nms_limit < A) ? pre_nms_limit : A;
  const float window[4] = {0.0f, 0.0f, 1.0f, 1.0f};
#pragma omp parallel for schedule(dynamic, 1)
  for (int32_t b = 0; b < B; ++b) {
    int32_t* ix = (int32_t*)malloc(sizeof(int32_t) * (size_t)(K + 1));
    float* sc = (float*)malloc(sizeof(float) * (size_t)(K + 1));
    float* clipped = (float*)malloc(sizeof(float) * 4 * (size_t)(K + 1));
    int32_t* keep = (int32_t*)malloc(sizeof(int32_t) * (size_t)(N + 1));
    /* scores = probs[:,:,1]; ix = top_k(scores, K).indices   (:153-169) */
    orc_topk(probs + (int64_t)b * A * 2 + 1, 1, A, 0, 2, K, ix, sc);
    for (int32_t k = 0; k < K; ++k) {
      const int64_t src = ((int64_t)b * A + ix[k]) * 4;
      float d[4], dec[4];
      for (int c = 0; c < 4; ++c) d[c] = bbox[src + c] * stddev[c];      /* :157 */
      decode_one(anchors + src, d, dec);                                  /* :179 */
      clip_one(dec, window, clipped + 4 * k);                             /* :183 */
      const int64_t dst = ((int64_t)b * K + k);
      if (ix_out) ix_out[dst] = ix[k];
      if (scores_out) scores_out[dst] = sc[k];
      for (int c = 0; c < 4; ++c) {
        if (delta_out) delta_out[dst * 4 + c] = d[c];
        if (anchors_out) anchors_out[dst * 4 + c] = anchors[src + c];
        if (decoded_out) decoded_out[dst * 4 + c] = dec[c];
        if (clipped_out) clipped_out[dst * 4 + c] = clipped[4 * k + c];
      }
    }
    /* per image NMS + zero pad (:218-247) */
    const int32_t cnt = orc_nms(clipped, sc, K, N, nms_thr, keep);
    float* p = proposals + (int64_t)b * N * 4;
    memset(p, 0, sizeof(float) * 4 * (size_t)N);
    for (int32_t j = 0; j < cnt; ++j) memcpy(p + 4 * j, clipped + 4 * (int64_t)keep[j], 4 * sizeof(float));
    if (keep_out) for (int32_t j = 0; j < N; ++j) keep_out[(int64_t)b * N + j] = (j < cnt) ? keep[j] : -1;
    if (num_kept_out) num_kept_out[b] = cnt;
    free(ix); free(sc); free(clipped); free(keep);
  }
}

/* ------------------------------------------------------------------------- */
/* BuildDetectionTargets, data_processor.py:430-658 (one image).                */
static inline float target_iou(const float* p, const float* g) { /* get_iou_tf :473-510 */
  const float p_area = (p[2] - p[0]) * (p[3] - p[1]);
  const float g_area = (g[2] - g[0]) * (g[3] - g[1]);
  const float iy1 = f_max(p[0], g[0]), ix1 = f_max(p[1], g[1]);
  const float iy2 = f_min(p[2], g[2]), ix2 = f_min(p[3], g[3]);
  const float inter = f_max(iy2 - iy1, 0.0f) * f_max(ix2 - ix1, 0.0f);
  return inter / ((p_area + g_area) - inter);
}
ORC_API float orc_target_iou(const float* p, const float* g) { return target_iou(p, g); }

/* box_refinement_tf :443-471 then "/= stddev" :616 */
static inline void refine_one(const float* box, const float* gt, const float* stddev, float* o) {
  const float height = box[2] - box[0];
  const float width = box[3] - box[1];
  const float center_y = box[0] + 0.5f * height;
  const float center_x = box[1] + 0.5f * width;
  const float gt_height = gt[2] - gt[0];
  const float gt_width = gt[3] - gt[1];
  const float gt_center_y = gt[0] + 0.5f * gt_height;
  const float gt_center_x = gt[1] + 0.5f * gt_width;
  o[0] = ((gt_center_y - center_y) / height) / stddev[0];
  o[1] = ((gt_center_x - center_x) / width) / stddev[1];
  o[2] = f_log(gt_height / height) / stddev[2];
  o[3] = f_log(gt_width / width) / stddev[3];
}

/* counts_out[6] = n_prop, n_gt, n_pos_all, n_neg_all, pos_count, neg_count.
 * Optional outputs may be NULL. iou_out is [N,G] with compacted rows/cols filled.
 * Returns 0, or -1 if pos_count + neg_count exceeds R (cannot be represented in [R,*]). */
ORC_API int32_t orc_detection_targets(const float* proposals /*[N,4]*/, const int32_t* gt_class_ids /*[G]*/,
                                      const float* gt_boxes /*[G,4]*/, int32_t N, int32_t G,
                                      const int32_t* perm_pos /*[N]*/, const int32_t* perm_neg /*[N]*/,
                                      int32_t R, const float* stddev,
                                      float* rois /*[R,4]*/, int32_t* roi_cls /*[R]*/, float* roi_deltas /*[R,4]*/,
                                      float* iou_out, float* iou_max_out /*[N]*/, int32_t* pos_all_out /*[N]*/,
                                      int32_t* neg_all_out /*[N]*/, int32_t* counts_out /*[6]*/,
                                      int32_t* sampled_pos_out /*[R]*/, int32_t* sampled_neg_out /*[R]*/,
                                      int32_t* assign_out /*[R]*/) {
  int32_t* prop_src = (int32_t*)malloc(sizeof(int32_t) * (size_t)(N + 1));
  int32_t* gt_src = (int32_t*)malloc(sizeof(int32_t) * (size_t)(G + 1));
  int32_t n_prop = 0, n_gt = 0;
  /* :564-571 strip zero padding (cast-to-bool of sum|coords|; NaN counts as non-zero) */
  for (int32_t i = 0; i < N; ++i) {
    const float* p = proposals + 4 * (int64_t)i;
    const float s = ((fabsf(p[0]) + fabsf(p[1])) + fabsf(p[2])) + fabsf(p[3]);
    if (s != 0.0f) prop_src[n_prop++] = i;
  }
  for (int32_t j = 0; j < G; ++j) if (gt_class_ids[j] != 0) gt_src[n_gt++] = j;

  float* iou_max = (float*)malloc(sizeof(float) * (size_t)(n_prop + 1));
  int32_t* iou_arg = (int32_t*)malloc(sizeof(int32_t) * (size_t)(n_prop + 1));
  int32_t* pos = (int32_t*)malloc(sizeof(int32_t) * (size_t)(n_prop + 1));
  int32_t* neg = (int32_t*)malloc(sizeof(int32_t) * (size_t)(n_prop + 1));
  int32_t n_pos = 0, n_neg = 0;
  for (int32_t i = 0; i < n_prop; ++i) {           /* :576-583 */
    float best = -INFINITY; int32_t arg = 0;
    for (int32_t j = 0; j < n_gt; ++j) {
      const float v = target_iou(proposals + 4 * (int64_t)prop_src[i], gt_boxes + 4 * (int64_t)gt_src[j]);
      if (iou_out) iou_out[(int64_t)i * G + j] = v;
      if (v > best) { best = v; arg = j; }         /* first maximum */
    }
    iou_max[i] = best; iou_arg[i] = arg;
    if (iou_max_out) iou_max_out[i] = best;
    if (best >= 0.5f) pos[n_pos++] = i;
    if (best < 0.5f) neg[n_neg++] = i;
  }
  if (pos_all_out) for (int32_t i = 0; i < N; ++i) pos_all_out[i] = (i < n_pos) ? pos[i] : -1;
  if (neg_all_out) for (int32_t i = 0; i < N; ++i) neg_all_out[i] = (i < n_neg) ? neg[i] : -1;

  /* :586-597 sampling. tf.random_shuffle is replaced by the explicit permutations. */
  const int32_t num_pos_inst = (int32_t)((double)R * 0.33);
  const int32_t pos_count = (n_pos < num_pos_inst) ? n_pos : num_pos_inst;
  const float inv = (float)(1.0 / 0.33);
  int32_t neg_cnt = f_to_i32(inv * (float)pos_count) - pos_count;
  if (neg_cnt < 0) neg_cnt = 0;
  const int32_t neg_count = (n_neg < neg_cnt) ? n_neg : neg_cnt;
  if (counts_out) {
    counts_out[0] = n_prop; counts_out[1] = n_gt; counts_out[2] = n_pos; counts_out[3] = n_neg;
    counts_out[4] = pos_count; counts_out[5] = neg_count;
  }
  int32_t rc = 0;
  memset(rois, 0, sizeof(float) * 4 * (size_t)R);
  memset(roi_cls, 0, sizeof(int32_t) * (size_t)R);
  memset(roi_deltas, 0, sizeof(float) * 4 * (size_t)R);
  if (sampled_pos_out) for (int32_t i = 0; i < R; ++i) sampled_pos_out[i] = -1;
  if (sampled_neg_out) for (int32_t i = 0; i < R; ++i) sampled_neg_out[i] = -1;
  if (assign_out) for (int32_t i = 0; i < R; ++i) assign_out[i] = -1;
  if (pos_count + neg_count > R) rc = -1;
  else {
    int32_t taken = 0;
    for (int32_t t = 0; t < N && taken < pos_count; ++t) {
      const int32_t q = perm_pos[t];
      if (q < 0 || q >= n_pos) continue;
      const int32_t idx = pos[q];                  /* index in compacted space */
      /* :600 gathers from the UN-compacted proposals with compacted indices */
      const float* box = proposals + 4 * (int64_t)idx;
      const int32_t g = gt_src[iou_arg[idx]];      /* :609-612 */
      memcpy(rois + 4 * (int64_t)taken, box, 4 * sizeof(float));
      roi_cls[taken] = gt_class_ids[g];
      refine_one(box, gt_boxes + 4 * (int64_t)g, stddev, roi_deltas + 4 * (int64_t)taken);
      if (sampled_pos_out) sampled_pos_out[taken] = idx;
      if (assign_out) assign_out[taken] = iou_arg[idx];
      taken++;
    }
    int32_t ntaken = 0;
    for (int32_t t = 0; t < N && ntaken < neg_count; ++t) {
      const int32_t q = perm_neg[t];
      if (q < 0 || q >= n_neg) continue;
      const int32_t idx = neg[q];
      memcpy(rois + 4 * (int64_t)(pos_count + ntaken), proposals + 4 * (int64_t)idx, 4 * sizeof(float));
      if (sampled_neg_out) sampled_neg_out[ntaken] = idx;
      ntaken++;
    }
  }
  free(prop_src); free(gt_src); free(iou_max); free(iou_arg); free(pos); free(neg);
  return rc;
}

/* ------------------------------------------------------------------------- */
/* DetectionLayer.build, detection.py:80-260 (one image per OpenMP task).
 * window [B,4] is already normalised. detections [B,M,6]. Optional outputs NULL-able. */
ORC_API void orc_detection_forward(const float* proposals /*[B,N,4]*/, const float* probs /*[B,N,C]*/,
                                   const float* bbox /*[B,N,C,4]*/, const float* window /*[B,4]*/,
                                   int32_t B, int32_t N, int32_t C, const float* stddev,
                                   float min_conf, float nms_thr, int32_t M, float* detections,
                                   int32_t* class_ids_out /*[B,N]*/, float* class_scores_out /*[B,N]*/,
                                   float* refined_out /*[B,N,4]*/, float* clipped_out /*[B,N,4]*/,
                                   int32_t* keep_mask_out /*[B,N]*/, int32_t* nms_keep_mask_out /*[B,N]*/) {
#pragma omp parallel for schedule(dynamic, 1)
  for (int32_t b = 0; b < B; ++b) {
    int32_t* cls = (int32_t*)malloc(sizeof(int32_t) * (size_t)(N + 1));
    float* score = (float*)malloc(sizeof(float) * (size_t)(N + 1));
    float* clipped = (float*)malloc(sizeof(float) * 4 * (size_t)(N + 1));
    uint8_t* keep = (uint8_t*)calloc((size_t)(N + 1), 1);
    uint8_t* nms_keep = (uint8_t*)calloc((size_t)(N + 1), 1);
    int32_t* member = (int32_t*)malloc(sizeof(int32_t) * (size_t)(N + 1));
    float* mboxes = (float*)malloc(sizeof(float) * 4 * (size_t)(N + 1));
    float* mscores = (float*)malloc(sizeof(float) * (size_t)(N + 1));
    int32_t* mkeep = (int32_t*)malloc(sizeof(int32_t) * (size_t)(M + 1));
    for (int32_t n = 0; n < N; ++n) {
      const int64_t r = (int64_t)b * N + n;
      const float* p = probs + r * C;
      int32_t arg = 0; float best = p[0];                       /* :115 argmax, first max */
      for (int32_t c = 1; c < C; ++c) if (p[c] > best) { best = p[c]; arg = c; }
      cls[n] = arg; score[n] = p[arg];                           /* :129 */
      float d[4], ref[4];
      for (int c = 0; c < 4; ++c) d[c] = bbox[(r * C + arg) * 4 + c] * stddev[c];  /* :117,:130 */
      decode_one(proposals + r * 4, d, ref);                     /* :133 */
      clip_one(ref, window + 4 * (int64_t)b, clipped + 4 * (int64_t)n);  /* :147 */
      keep[n] = (uint8_t)((arg > 0) && (score[n] > min_conf));   /* :152-158 */
      if (class_ids_out) class_ids_out[r] = arg;
      if (class_scores_out) class_scores_out[r] = score[n];
      for (int c = 0; c < 4; ++c) {
        if (refined_out) refined_out[r * 4 + c] = ref[c];
        if (clipped_out) clipped_out[r * 4 + c] = clipped[4 * n + c];
      }
      if (keep_mask_out) keep_mask_out[r] = keep[n];
    }
    /* per-class NMS (:167-204). Class visiting order does not affect the result. */
    for (int32_t c = 1; c < C; ++c) {
      int32_t m = 0;
      for (int32_t n = 0; n < N; ++n) if (keep[n] && cls[n] == c) {
        member[m] = n; mscores[m] = score[n];
        memcpy(mboxes + 4 * (int64_t)m, clipped + 4 * (int64_t)n, 4 * sizeof(float)); m++;
      }
      if (m == 0) continue;
      const int32_t cnt = orc_nms(mboxes, mscores, m, M, nms_thr, mkeep);
      for (int32_t j = 0; j < cnt; ++j) nms_keep[member[mkeep[j]]] = 1;
    }
    /* :207-221 ascending ROI index list -> top_k(score) with ties to the lower index */
    uint64_t* order = (uint64_t*)malloc(sizeof(uint64_t) * (size_t)(N + 1));
    int32_t total = 0;
    for (int32_t n = 0; n < N; ++n) {
      if (nms_keep_mask_out) nms_keep_mask_out[(int64_t)b * N + n] = nms_keep[n];
      if (nms_keep[n]) order[total++] = composite_key(score[n], (uint32_t)n);
    }
    qsort(order, (size_t)total, sizeof(uint64_t), cmp_u64_desc);
    const int32_t num_keep = (total < M) ? total : M;
    float* det = detections + (int64_t)b * M * 6;
    memset(det, 0, sizeof(float) * 6 * (size_t)M);               /* :234-235 */
    for (int32_t j = 0; j < num_keep; ++j) {                    /* :226-230 */
      const int32_t n = (int32_t)composite_index(order[j]);
      memcpy(det + 6 * j, clipped + 4 * (int64_t)n, 4 * sizeof(float));
      det[6 * j + 4] = (float)cls[n];
      det[6 * j + 5] = score[n];
    }
    free(order); free(cls); free(score); free(clipped); free(keep); free(nms_keep);
    free(member); free(mboxes); free(mscores); free(mkeep);
  }
}

/* ------------------------------------------------------------------------- */
/* Anchors: utils.py:230-353 (fp64, ratio fastest, then x, y, level).           */
typedef struct {
  int32_t num_levels, num_ratios;
  double scales[8], ratios[8];
  int32_t fmap_h[8], fmap_w[8], fmap_stride[8];
  int32_t anchor_stride, image_h, image_w;
} orc_anchor_spec;

ORC_API int64_t orc_anchor_count(const orc_anchor_spec* s) {
  int64_t total = 0;
  for (int32_t l = 0; l < s->num_levels; ++l) {
    const int64_t ny = (s->fmap_h[l] + s->anchor_stride - 1) / s->anchor_stride;
    const int64_t nx = (s->fmap_w[l] + s->anchor_stride - 1) / s->anchor_stride;
    total += ny * nx * s->num_ratios;
  }
  return total;
}
/* pixel [A,4] f64 (gen_anchors_pixel_coord) and/or norm [A,4] f32 (gen_anchors + norm_boxes :181-196). */
ORC_API void orc_gen_anchors(const orc_anchor_spec* s, double* pixel, float* norm) {
  int64_t o = 0;
  const double scale_n[4] = {(double)(s->image_h - 1), (double)(s->image_w - 1),
                             (double)(s->image_h - 1), (double)(s->image_w - 1)};
  const double shift_n[4] = {0, 0, 1, 1};
  for (int32_t l = 0; l < s->num_levels; ++l) {
    const int32_t ny = (s->fmap_h[l] + s->anchor_stride - 1) / s->anchor_stride;
    const int32_t nx = (s->fmap_w[l] + s->anchor_stride - 1) / s->anchor_stride;
    for (int32_t y = 0; y < ny; ++y)
      for (int32_t x = 0; x < nx; ++x)
        for (int32_t r = 0; r < s->num_ratios; ++r, ++o) {
          const double sq = sqrt(s->ratios[r]);
          const double h = s->scales[l] / sq;
          const double w = s->scales[l] * sq;
          const double cy = (double)((int64_t)y * s->anchor_stride * s->fmap_stride[l]);
          const double cx = (double)((int64_t)x * s->anchor_stride * s->fmap_stride[l]);
          const double box[4] = {cy - 0.5 * h, cx - 0.5 * w, cy + 0.5 * h, cx + 0.5 * w};
          for (int c = 0; c < 4; ++c) {
            if (pixel) pixel[o * 4 + c] = box[c];
            if (norm) norm[o * 4 + c] = (float)((box[c] - shift_n[c]) / scale_n[c]);
          }
        }
  }
}

/* ------------------------------------------------------------------------- */
/* Faster R-CNN numpy proposal layer, FasterRCNN/building_blocks/proposals.py.
 * fp64 like the reference's numpy code. Boxes are (x1,y1,x2,y2) pixels, +1 widths. */
ORC_API void orc_frcnn_decode(const double* anchors, const double* deltas, int64_t n, double* out) {
  for (int64_t i = 0; i < n; ++i) {               /* corner_pixels_to_center_inv :286-309 */
    const double* a = anchors + 4 * i; const double* d = deltas + 4 * i; double* o = out + 4 * i;
    const double aw = a[2] - a[0] + 1, ah = a[3] - a[1] + 1;
    const double acx = a[0] + aw / 2, acy = a[1] + ah / 2;
    const double pcx = d[0] * aw + acx, pcy = d[1] * ah + acy;
    const double pw = exp(d[2]) * aw, ph = exp(d[3]) * ah;
    o[0] = pcx - pw / 2; o[1] = pcy - ph / 2; o[2] = pcx + pw / 2; o[3] = pcy + ph / 2;
  }
}
static inline double d_min(double a, double b) { return (b < a) ? b : a; }
static inline double d_max(double a, double b) { return (a < b) ? b : a; }

/* greedy NMS of proposals.py:127-169 on boxes already in visiting order.
 * Returns the number kept (<= max_out) and their positions. */
ORC_API int32_t orc_frcnn_nms_sorted(const double* boxes, int32_t n, double thr, int32_t max_out, int32_t* keep) {
  uint8_t* sup = (uint8_t*)calloc((size_t)(n + 1), 1);
  int32_t cnt = 0;
  for (int32_t i = 0; i < n; ++i) {
    if (sup[i]) continue;
    if (cnt < max_out) keep[cnt] = i;
    cnt++;
    const double* bi = boxes + 4 * (int64_t)i;
    const double iarea = (bi[2] - bi[0] + 1) * (bi[3] - bi[1] + 1);
    for (int32_t j = i + 1; j < n; ++j) {
      if (sup[j]) continue;
      const double* bj = boxes + 4 * (int64_t)j;
      const double xx1 = d_max(bi[0], bj[0]), yy1 = d_max(bi[1], bj[1]);
      const double xx2 = d_min(bi[2], bj[2]), yy2 = d_min(bi[3], bj[3]);
      const double w = d_max(0.0, xx2 - xx1 + 1), h = d_max(0.0, yy2 - yy1 + 1);
      const double inter = w * h;
      const double jarea = (bj[2] - bj[0] + 1) * (bj[3] - bj[1] + 1);
      const double ovr = inter / (iarea + jarea - inter);
      if (ovr >= thr) sup[j] = 1;
    }
  }
  free(sup);
  return (cnt < max_out) ? cnt : max_out;
}

static inline uint64_t d_key(double s) {   /* score_key's order: -0 == +0, every NaN above +inf */
  uint64_t b;
  if (s != s) return 0xFFFFFFFFFFFFFFFFull;
  s = s + 0.0; memcpy(&b, &s, 8);
  return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}
typedef struct { uint64_t key; int32_t idx; } dk_t;
static int cmp_dk_desc(const void* a, const void* b) {
  const dk_t* x = (const dk_t*)a; const dk_t* y = (const dk_t*)b;
  if (x->key != y->key) return (x->key < y->key) - (x->key > y->key);
  return (x->idx > y->idx) - (x->idx < y->idx);
}

/* Proposals.build :392-512 with the INTENDED top-N (flattened stable descending order).
 * probs [h,w,2*na] (fg = channels [:na]), bbox [h,w,4*na]; out [post,5] f32 rows (0,x1,y1,x2,y2).
 * Returns number of proposals. */
ORC_API int32_t orc_frcnn_proposals(const double* probs, const double* bbox, int32_t h, int32_t w,
                                    int32_t na, const double* base_anchors, int32_t feat_stride,
                                    int32_t image_h, int32_t image_w, int32_t min_hw,
                                    int32_t pre_n, int32_t post_n, double thr, float* out) {
  const int64_t total = (int64_t)h * w * na;
  double* boxes = (double*)malloc(sizeof(double) * 4 * (size_t)total);
  dk_t* order = (dk_t*)malloc(sizeof(dk_t) * (size_t)total);
  int64_t m = 0;
  for (int64_t pos = 0; pos < (int64_t)h * w; ++pos) {
    const double sx = (double)((pos % w) * feat_stride), sy = (double)((pos / w) * feat_stride);
    for (int32_t a = 0; a < na; ++a) {
      const int64_t i = pos * na + a;
      const double anc[4] = {base_anchors[4 * a] + sx, base_anchors[4 * a + 1] + sy,
                             base_anchors[4 * a + 2] + sx, base_anchors[4 * a + 3] + sy};
      double bx[4];
      orc_frcnn_decode(anc, bbox + 4 * i, 1, bx);
      bx[0] = d_max(d_min(bx[0], (double)(image_w - 1)), 0.0);   /* clip_boxes :335-338 */
      bx[1] = d_max(d_min(bx[1], (double)(image_h - 1)), 0.0);
      bx[2] = d_max(d_min(bx[2], (double)(image_w - 1)), 0.0);
      bx[3] = d_max(d_min(bx[3], (double)(image_h - 1)), 0.0);
      if ((bx[2] - bx[0] + 1 >= (double)min_hw) && (bx[3] - bx[1] + 1 >= (double)min_hw)) {  /* :342-345 */
        memcpy(boxes + 4 * m, bx, sizeof(bx));
        order[m].key = d_key(probs[pos * 2 * na + a]);
        order[m].idx = (int32_t)m;
        m++;
      }
    }
  }
  qsort(order, (size_t)m, sizeof(dk_t), cmp_dk_desc);
  const int32_t npre = (int32_t)((m < pre_n) ? m : pre_n);
  double* sorted = (double*)malloc(sizeof(double) * 4 * (size_t)(npre + 1));
  for (int32_t i = 0; i < npre; ++i) memcpy(sorted + 4 * (int64_t)i, boxes + 4 * (int64_t)order[i].idx, 4 * sizeof(double));
  int32_t* keep = (int32_t*)malloc(sizeof(int32_t) * (size_t)(post_n + 1));
  const int32_t cnt = orc_frcnn_nms_sorted(sorted, npre, thr, post_n, keep);
  memset(out, 0, sizeof(float) * 5 * (size_t)post_n);
  for (int32_t j = 0; j < cnt; ++j) {
    out[5 * j] = 0.0f;
    for (int c = 0; c < 4; ++c) out[5 * j + 1 + c] = (float)sorted[4 * (int64_t)keep[j] + c];
  }
  free(boxes); free(order); free(sorted); free(keep);
  return cnt;
}

/* roi_pool, FasterRCNN/building_blocks/fastrcnn.py:22-70: crop 14x14 then 2x2 max pool. */
ORC_API void orc_roi_pool(const float* fmap, int32_t B, int32_t H, int32_t W, int32_t D,
                          const float* proposals /*[n,5]*/, int32_t n, float image_h, float image_w,
                          float* out /*[n,7,7,D]*/) {
  float* boxes = (float*)malloc(sizeof(float) * 4 * (size_t)(n + 1));
  int32_t* bi = (int32_t*)malloc(sizeof(int32_t) * (size_t)(n + 1));
  float* crop = (float*)malloc(sizeof(float) * (size_t)(n + 1) * 14 * 14 * (size_t)D);
  for (int32_t i = 0; i < n; ++i) {
    const float* p = proposals + 5 * (int64_t)i;
    bi[i] = (int32_t)p[0];
    boxes[4 * i + 0] = p[2] / image_h; boxes[4 * i + 1] = p[1] / image_w;
    boxes[4 * i + 2] = p[4] / image_h; boxes[4 * i + 3] = p[3] / image_w;
  }
  memset(crop, 0, sizeof(float) * (size_t)(n + 1) * 14 * 14 * (size_t)D);
  orc_crop_and_resize(fmap, B, H, W, D, boxes, bi, n, 14, 14, 0.0f, crop);
  for (int32_t i = 0; i < n; ++i)
    for (int32_t y = 0; y < 7; ++y)
      for (int32_t x = 0; x < 7; ++x)
        for (int32_t d = 0; d < D; ++d) {
          const float* c = crop + (((int64_t)i * 14 + 2 * y) * 14 + 2 * x) * D + d;
          float v = c[0];
          v = f_max(v, c[D]); v = f_max(v, c[14 * (int64_t)D]); v = f_max(v, c[14 * (int64_t)D + D]);
          out[(((int64_t)i * 7 + y) * 7 + x) * D + d] = v;
        }
  free(boxes); free(bi); free(crop);
}
