// rpn_targets.cu — RPN target builder: PreprareTrainData.build_rpn_targets (data_processor.py:173-294) with
// utils.intersection_over_union (utils.py:32-40), batched over images. SURVEY.md §8(f) rank 1: the step in front of
// the detection-head path in training (anchors x GT IoU, 261,888 x <=100 per image).
//
// The reference is numpy float64 throughout, so every kernel here computes in fp64 and the labels are bit-exact:
//   rpn_anchor_best_kernel : one thread per anchor, GT boxes in shared memory -> max IoU / first argmax per anchor; for
//                            G <= 256 also the per-CTA partial of the first argmax per GT ("best anchor" rule :232),
//                            folded by rpn_gt_reduce_kernel. An fp32 sign test on outward-rounded boxes skips the
//                            disjoint pairs (IoU exactly 0) before any fp64 arithmetic.
//   rpn_gt_best_kernel     : G > 256 only: one CTA per (GT, image) over all anchors
//   rpn_label_kernel       : -1 (< 0.3) / +1 (>= 0.7 or best anchor of a GT) / 0                       (:224-238)
//   rpn_count / rpn_compact / rpn_perm<count> / rpn_perm<apply> : balance to max_rpn_targets (:242-262), 1024 anchors
//                            per CTA, with the two np.random.choice draws replaced by explicit permutations (the list
//                            element at position q is dropped for the first `extra` entries q of the permutation with
//                            q < len(list))
//   rpn_emit_kernel        : the fp64 box deltas of the surviving positives (:265-291).
#include "common.cuh"

namespace od {

constexpr int kRpnThreads = 256;
constexpr int kRpnWarps = kRpnThreads / 32;
constexpr int kFusedMaxGt = 256;   // fused per-GT arg-max: 8 warps x G x 12 B of shared memory
constexpr int kChunk = 4 * kRpnThreads;   // anchors (or permutation entries) per CTA in the subsampling kernels
constexpr int kRpnSubThreads = 1024;

// utils.intersection_over_union: box = GT, boxes = anchors; union = (box_area + boxes_area) - intersection.
__device__ __forceinline__ double rpn_iou(const double* g, double g_area, double a0, double a1, double a2, double a3, double a_area) {
  const double y1 = fmax(g[0], a0), y2 = fmin(g[2], a2);
  const double x1 = fmax(g[1], a1), x2 = fmin(g[3], a3);
  const double inter = fmax(x2 - x1, 0.0) * fmax(y2 - y1, 0.0);
  // disjoint boxes: 0 / union is +-0 (the comparisons below treat both alike); skips the fp64 divide for ~99 % of pairs
  if (inter == 0.0) return 0.0;
  const double uni = g_area + a_area - inter;
  return inter / uni;
}

// Conservative fp32 copy of an fp64 box: mins rounded down, maxes rounded up. If the exact boxes overlap with positive
// width and height, the rounded ones do too, so four fp32 sign tests are a superset filter for "IoU > 0"; disjoint
// pairs have IoU exactly 0 in the reference's arithmetic and never reach the fp64 code.
__device__ __forceinline__ float4 conservative_f32(double y1, double x1, double y2, double x2) {
  return make_float4(__double2float_rd(y1), __double2float_rd(x1), __double2float_ru(y2), __double2float_ru(x2));
}
__device__ __forceinline__ bool may_overlap(float4 a, float4 g) {
  const uint32_t sgn = __float_as_uint(g.x - a.z) & __float_as_uint(a.x - g.z) & __float_as_uint(g.y - a.w) &
                       __float_as_uint(a.y - g.w);
  return (int32_t)sgn < 0;
}

// FUSED (G <= kFusedMaxGt): the same pass also tracks, per GT box, the best anchor of this CTA's 256 anchors — a warp
// arg-max whenever some lane has IoU > 0 (a few percent of the (warp, GT) pairs), one private row of shared memory per
// warp — and writes one (IoU, anchor) partial per (image, GT, CTA); rpn_gt_reduce_kernel folds the partials.
// Otherwise rpn_gt_best_kernel re-walks the anchors per GT.
template <bool FUSED>
__global__ void __launch_bounds__(kRpnThreads)
rpn_anchor_best_kernel(const double* __restrict__ anchors, int A, const double* __restrict__ gt, const int32_t* __restrict__ gt_count,
                       int G, double* __restrict__ iou_max, int32_t* __restrict__ iou_arg, float4* __restrict__ anchors_c,
                       double* __restrict__ part_v, int32_t* __restrict__ part_i) {
  pdl_prologue();
  extern __shared__ double s_gt[];   // [G][5]: y1,x1,y2,x2,area; [G] float4 conservative copies; FUSED: [warps][G] best IoU, anchor
  float4* s_gc = reinterpret_cast<float4*>(s_gt + (size_t)G * 5 + (G & 1));
  double* s_wv = reinterpret_cast<double*>(s_gc + G);
  int32_t* s_wi = reinterpret_cast<int32_t*>(s_wv + (size_t)kRpnWarps * G);
  const int b = blockIdx.y;
  const int ng = min(gt_count[b], G);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int a = blockIdx.x * kRpnThreads + threadIdx.x;
  const bool valid = a < A;
  for (int j = threadIdx.x; j < ng; j += kRpnThreads) {
    const double* g = gt + ((int64_t)b * G + j) * 4;
    s_gt[j * 5 + 0] = g[0]; s_gt[j * 5 + 1] = g[1]; s_gt[j * 5 + 2] = g[2]; s_gt[j * 5 + 3] = g[3];
    s_gt[j * 5 + 4] = (g[2] - g[0]) * (g[3] - g[1]);
    s_gc[j] = conservative_f32(g[0], g[1], g[2], g[3]);
  }
  if (FUSED) {
    // all-zero column: np.argmax returns the first anchor; a warp past the end of the anchors never wins
    const int first = a - lane;
    for (int j = lane; j < ng; j += 32) {
      s_wv[warp * G + j] = (first < A) ? 0.0 : -1.0;
      s_wi[warp * G + j] = first;
    }
  }
  __syncthreads();
  if (!FUSED && !valid) return;
  double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
  float4 ac = make_float4(INFINITY, INFINITY, -INFINITY, -INFINITY);   // overlaps nothing
  if (valid) {
    a0 = anchors[4 * (int64_t)a]; a1 = anchors[4 * (int64_t)a + 1]; a2 = anchors[4 * (int64_t)a + 2]; a3 = anchors[4 * (int64_t)a + 3];
    ac = conservative_f32(a0, a1, a2, a3);
    if (b == 0) anchors_c[a] = ac;   // for rpn_gt_best_kernel
  }
  const double a_area = (a2 - a0) * (a3 - a1);
  double best = 0.0;   // no GT: every anchor is background; all-disjoint: IoU 0 with the first GT (np.argmax)
  int arg = 0;
  for (int j = 0; j < ng; ++j) {
    const bool cand = may_overlap(ac, s_gc[j]);   // otherwise IoU is exactly 0: cannot beat `best` (>= 0, strict compare)
    if (!FUSED && !cand) continue;
    double v = 0.0;
    bool hit = false;
    if (cand) {
      v = rpn_iou(&s_gt[j * 5], s_gt[j * 5 + 4], a0, a1, a2, a3, a_area);
      hit = v > 0.0;
      if (v > best) {   // np.argmax: first maximum
        best = v;
        arg = j;
      }
    }
    if (FUSED && __any_sync(0xffffffffu, hit)) {
      double mv = v;
      int mi = a;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, mv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, mi, o);
        if (ov > mv || (ov == mv && oi < mi)) {
          mv = ov;
          mi = oi;
        }
      }
      if (lane == 0) {
        s_wv[warp * G + j] = mv;
        s_wi[warp * G + j] = mi;
      }
    }
  }
  if (valid) {
    iou_max[(int64_t)b * A + a] = best;
    iou_arg[(int64_t)b * A + a] = arg;
  }
  if (FUSED) {
    __syncthreads();
    for (int j = threadIdx.x; j < ng; j += kRpnThreads) {
      double bv = s_wv[j];
      int bi = s_wi[j];
      for (int w = 1; w < kRpnWarps; ++w)
        if (s_wv[w * G + j] > bv) {   // warps ascend in anchor index: a tie keeps the earlier one
          bv = s_wv[w * G + j];
          bi = s_wi[w * G + j];
        }
      part_v[((int64_t)b * G + j) * gridDim.x + blockIdx.x] = bv;
      part_i[((int64_t)b * G + j) * gridDim.x + blockIdx.x] = bi;
    }
  }
}

// Folds the per-CTA partials of the fused kernel: first maximum in anchor order.
__global__ void __launch_bounds__(kRpnThreads)
rpn_gt_reduce_kernel(const double* __restrict__ part_v, const int32_t* __restrict__ part_i, int nchunk,
                     const int32_t* __restrict__ gt_count, int G, int32_t* __restrict__ gt_best) {
  pdl_prologue();
  __shared__ double s_v[kRpnThreads];
  __shared__ int32_t s_i[kRpnThreads];
  const int j = blockIdx.x, b = blockIdx.y;
  if (j >= min(gt_count[b], G)) {
    if (threadIdx.x == 0) gt_best[(int64_t)b * G + j] = -1;
    return;
  }
  const double* pv = part_v + ((int64_t)b * G + j) * nchunk;
  const int32_t* pi = part_i + ((int64_t)b * G + j) * nchunk;
  double best = -1.0;
  int arg = 0x7fffffff;
  for (int c = threadIdx.x; c < nchunk; c += kRpnThreads)
    if (pv[c] > best) {
      best = pv[c];
      arg = pi[c];
    }
  s_v[threadIdx.x] = best;
  s_i[threadIdx.x] = arg;
  __syncthreads();
  for (int o = kRpnThreads / 2; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      const double ov = s_v[threadIdx.x + o];
      const int oi = s_i[threadIdx.x + o];
      if (ov > s_v[threadIdx.x] || (ov == s_v[threadIdx.x] && oi < s_i[threadIdx.x])) {
        s_v[threadIdx.x] = ov;
        s_i[threadIdx.x] = oi;
      }
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) gt_best[(int64_t)b * G + j] = (s_i[0] == 0x7fffffff) ? 0 : s_i[0];
}

__global__ void __launch_bounds__(kRpnThreads)
rpn_gt_best_kernel(const double* __restrict__ anchors, const float4* __restrict__ anchors_c, int A,
                   const double* __restrict__ gt, const int32_t* __restrict__ gt_count, int G, int32_t* __restrict__ gt_best) {
  pdl_prologue();
  __shared__ double s_v[kRpnThreads];
  __shared__ int32_t s_i[kRpnThreads];
  const int j = blockIdx.x, b = blockIdx.y;
  if (j >= min(gt_count[b], G)) {
    if (threadIdx.x == 0) gt_best[(int64_t)b * G + j] = -1;
    return;
  }
  const double* gp = gt + ((int64_t)b * G + j) * 4;
  const double g[4] = {gp[0], gp[1], gp[2], gp[3]};
  const double g_area = (g[2] - g[0]) * (g[3] - g[1]);
  const float4 gc = conservative_f32(g[0], g[1], g[2], g[3]);
  double best = -1.0;
  int arg = 0x7fffffff;
  for (int a = threadIdx.x; a < A; a += kRpnThreads) {
    double v = 0.0;   // disjoint: IoU is exactly 0
    if (may_overlap(__ldg(&anchors_c[a]), gc)) {
      const double a0 = anchors[4 * (int64_t)a], a1 = anchors[4 * (int64_t)a + 1], a2 = anchors[4 * (int64_t)a + 2],
                   a3 = anchors[4 * (int64_t)a + 3];
      v = rpn_iou(g, g_area, a0, a1, a2, a3, (a2 - a0) * (a3 - a1));
    }
    if (v > best) {   // ascending a per thread: the first maximum wins
      best = v;
      arg = a;
    }
  }
  s_v[threadIdx.x] = best;
  s_i[threadIdx.x] = arg;
  __syncthreads();
  for (int o = kRpnThreads / 2; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      const double ov = s_v[threadIdx.x + o];
      const int oi = s_i[threadIdx.x + o];
      if (ov > s_v[threadIdx.x] || (ov == s_v[threadIdx.x] && oi < s_i[threadIdx.x])) {
        s_v[threadIdx.x] = ov;
        s_i[threadIdx.x] = oi;
      }
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) gt_best[(int64_t)b * G + j] = (s_i[0] == 0x7fffffff) ? 0 : s_i[0];
}

__global__ void rpn_label_kernel(const double* __restrict__ iou_max, int64_t total, int32_t* __restrict__ cls) {
  pdl_prologue();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const double m = iou_max[i];
  cls[i] = (m >= 0.7) ? 1 : ((m < 0.3) ? -1 : 0);
}
__global__ void rpn_label_best_kernel(const int32_t* __restrict__ gt_best, int G, int A, int32_t* __restrict__ cls) {
  pdl_prologue();
  const int j = threadIdx.x + blockIdx.x * blockDim.x, b = blockIdx.y;
  if (j >= G) return;
  const int a = gt_best[(int64_t)b * G + j];
  OD_DBG_ASSERT(a < A, "best anchor of a GT box beyond the anchor count");
  if (a >= 0) cls[(int64_t)b * A + a] = 1;
}

constexpr int kCompactItems = 8;
// Stable compaction of {i in [0,n) : pred(i)} by a 1024-thread CTA, 8 consecutive elements per thread and round;
// emit(i, rank) for every selected i; returns the count. scratch: 33 ints of shared memory.
template <typename Pred, typename Emit>
__device__ int cta_compact(int n, Pred pred, Emit emit, int* scratch) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int base = 0;
  for (int t0 = 0; t0 < n; t0 += kCompactItems * kRpnSubThreads) {
    const int i0 = t0 + kCompactItems * tid;
    bool p[kCompactItems];
    int cnt = 0;
#pragma unroll
    for (int u = 0; u < kCompactItems; ++u) {
      p[u] = (i0 + u < n) && pred(i0 + u);
      cnt += p[u] ? 1 : 0;
    }
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += v;
    }
    if (lane == 31) scratch[warp] = incl;
    __syncthreads();
    if (warp == 0) {
      int w = scratch[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, w, o);
        if (lane >= o) w += v;
      }
      scratch[lane] = w;   // inclusive warp totals
    }
    __syncthreads();
    int r = base + (warp ? scratch[warp - 1] : 0) + incl - cnt;
#pragma unroll
    for (int u = 0; u < kCompactItems; ++u)
      if (p[u]) emit(i0 + u, r++);
    base += scratch[31];
    __syncthreads();
  }
  return base;
}

// ---- subsampling (:242-262), parallel over 1024-element chunks -----------------------------------------------------------
// cnt[b][chunk] = (#positives, #negatives) of the chunk; the prefix over chunks gives every CTA its base rank, so the
// ascending index lists np.where() returns are written by all CTAs at once. The np.random.choice replacement — "the
// list element at position q is dropped for the first `extra` entries q of the permutation with q < len(list)" — is the
// same count / prefix / apply over chunks of the permutation.
struct RpnTotals {
  int n_pos0, n_neg0, extra_pos, n_pos, extra_neg;
};
// Sum of the (x, y) pairs v[0..n) and of v[0..upto); every thread returns the same values. scratch: 32 ints.
__device__ void chunk_sums(const int2* __restrict__ v, int n, int upto, int2* total, int2* before, int* scratch) {
  int t[4] = {0, 0, 0, 0};
  for (int i = threadIdx.x; i < n; i += kRpnThreads) {
    const int2 c = v[i];
    t[0] += c.x;
    t[1] += c.y;
    if (i < upto) {
      t[2] += c.x;
      t[3] += c.y;
    }
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t[k] += __shfl_xor_sync(0xffffffffu, t[k], o);
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncthreads();   // scratch may still be in use by a previous call
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < 4; ++k) scratch[warp * 4 + k] = t[k];
  }
  __syncthreads();
  int r[4] = {0, 0, 0, 0};
  for (int w = 0; w < kRpnWarps; ++w) {
#pragma unroll
    for (int k = 0; k < 4; ++k) r[k] += scratch[w * 4 + k];
  }
  *total = make_int2(r[0], r[1]);
  *before = make_int2(r[2], r[3]);
}
__device__ __forceinline__ RpnTotals rpn_totals(int2 total, int max_targets) {
  RpnTotals t;
  t.n_pos0 = total.x;
  t.n_neg0 = total.y;
  t.extra_pos = t.n_pos0 - max_targets / 2;
  t.n_pos = t.extra_pos > 0 ? t.n_pos0 - t.extra_pos : t.n_pos0;
  t.extra_neg = t.n_neg0 - (max_targets - t.n_pos);
  return t;
}
// Exclusive scan of one packed (lo16, hi16) counter per thread over the CTA. scratch: kRpnWarps ints.
__device__ __forceinline__ int cta_scan_packed(int v, int* scratch, int* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int u = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += u;
  }
  __syncthreads();
  if (lane == 31) scratch[warp] = incl;
  __syncthreads();
  int off = 0, tot = 0;
  for (int w = 0; w < kRpnWarps; ++w) {
    const int c = scratch[w];
    if (w < warp) off += c;
    tot += c;
  }
  *total = tot;
  return off + incl - v;
}

__global__ void __launch_bounds__(kRpnThreads)
rpn_count_kernel(const int32_t* __restrict__ cls, int A, int2* __restrict__ cnt) {
  pdl_prologue();
  __shared__ int scratch[kRpnWarps];
  const int b = blockIdx.y, i0 = blockIdx.x * kChunk + 4 * threadIdx.x;
  const int32_t* c = cls + (int64_t)b * A;
  int v = 0;
#pragma unroll
  for (int u = 0; u < 4; ++u)
    if (i0 + u < A) {
      const int l = c[i0 + u];
      v += (l == 1) ? 1 : ((l == -1) ? (1 << 16) : 0);
    }
  int tot;
  cta_scan_packed(v, scratch, &tot);
  if (threadIdx.x == 0) cnt[(int64_t)b * gridDim.x + blockIdx.x] = make_int2(tot & 0xffff, tot >> 16);
}

// idx = np.where(cls == 1), np.where(cls == -1): ascending lists; also the per-image counts output.
__global__ void __launch_bounds__(kRpnThreads)
rpn_compact_kernel(const int32_t* __restrict__ cls, int A, const int2* __restrict__ cnt, int max_targets,
                   int32_t* __restrict__ list_pos, int32_t* __restrict__ list_neg, int32_t* __restrict__ counts) {
  pdl_prologue();
  __shared__ int scratch[32];
  const int b = blockIdx.y, i0 = blockIdx.x * kChunk + 4 * threadIdx.x;
  const int32_t* c = cls + (int64_t)b * A;
  int2 total, before;
  chunk_sums(cnt + (int64_t)b * gridDim.x, gridDim.x, blockIdx.x, &total, &before, scratch);
  int l[4];
  int v = 0;
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    l[u] = (i0 + u < A) ? c[i0 + u] : 0;
    v += (l[u] == 1) ? 1 : ((l[u] == -1) ? (1 << 16) : 0);
  }
  int tot;
  const int excl = cta_scan_packed(v, scratch, &tot);
  int rp = before.x + (excl & 0xffff), rn = before.y + (excl >> 16);
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    OD_DBG_ASSERT(rp <= A && rn <= A, "rank of a labelled anchor beyond the anchor count");
    if (l[u] == 1) list_pos[(int64_t)b * A + rp++] = i0 + u;
    if (l[u] == -1) list_neg[(int64_t)b * A + rn++] = i0 + u;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    const RpnTotals t = rpn_totals(total, max_targets);
    int32_t* o = counts + (int64_t)b * 4;
    o[0] = t.n_pos0;
    o[1] = t.n_neg0;
    o[2] = t.n_pos;
    o[3] = t.extra_neg > 0 ? t.n_neg0 - t.extra_neg : t.n_neg0;
  }
}

// APPLY = false: pcnt[b][chunk] = number of permutation entries of the chunk that address the list (q < len(list)).
// APPLY = true : entries whose rank among those is < extra clear the label of list[q].
template <bool APPLY>
__global__ void __launch_bounds__(kRpnThreads)
rpn_perm_kernel(const int32_t* __restrict__ perm_pos, const int32_t* __restrict__ perm_neg, int A, const int2* __restrict__ cnt,
                int2* __restrict__ pcnt, int max_targets, const int32_t* __restrict__ list_pos,
                const int32_t* __restrict__ list_neg, int32_t* __restrict__ cls) {
  pdl_prologue();
  __shared__ int scratch[32];
  const int b = blockIdx.y, i0 = blockIdx.x * kChunk + 4 * threadIdx.x;
  int2 total, before;
  chunk_sums(cnt + (int64_t)b * gridDim.x, gridDim.x, 0, &total, &before, scratch);
  const RpnTotals t = rpn_totals(total, max_targets);
  if (t.extra_pos <= 0 && t.extra_neg <= 0) {
    if (!APPLY && threadIdx.x == 0) pcnt[(int64_t)b * gridDim.x + blockIdx.x] = make_int2(0, 0);
    return;
  }
  int2 pbefore = make_int2(0, 0);
  if (APPLY) {
    int2 ptotal;
    chunk_sums(pcnt + (int64_t)b * gridDim.x, gridDim.x, blockIdx.x, &ptotal, &pbefore, scratch);
    if ((t.extra_pos <= 0 || pbefore.x >= t.extra_pos) && (t.extra_neg <= 0 || pbefore.y >= t.extra_neg)) return;
  }
  int qp[4], qn[4];
  int v = 0;
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    qp[u] = qn[u] = -1;
    if (i0 + u < A) {
      if (t.extra_pos > 0) qp[u] = perm_pos[(int64_t)b * A + i0 + u];
      if (t.extra_neg > 0) qn[u] = perm_neg[(int64_t)b * A + i0 + u];
    }
    if (qp[u] >= t.n_pos0) qp[u] = -1;
    if (qn[u] >= t.n_neg0) qn[u] = -1;
    v += (qp[u] >= 0 ? 1 : 0) + (qn[u] >= 0 ? (1 << 16) : 0);
  }
  int tot;
  const int excl = cta_scan_packed(v, scratch, &tot);
  if (!APPLY) {
    if (threadIdx.x == 0) pcnt[(int64_t)b * gridDim.x + blockIdx.x] = make_int2(tot & 0xffff, tot >> 16);
    return;
  }
  int rp = pbefore.x + (excl & 0xffff), rn = pbefore.y + (excl >> 16);
  int32_t* c = cls + (int64_t)b * A;
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    if (qp[u] >= 0 && rp++ < t.extra_pos) c[list_pos[(int64_t)b * A + qp[u]]] = 0;
    if (qn[u] >= 0 && rn++ < t.extra_neg) c[list_neg[(int64_t)b * A + qn[u]]] = 0;
  }
}

// Regression targets of the surviving positives, ascending anchor index (:256-291): one CTA per image walks the
// original positive list (short) and keeps the entries whose label is still 1.
__global__ void __launch_bounds__(kRpnSubThreads)
rpn_emit_kernel(const double* __restrict__ anchors, int A, const double* __restrict__ gt, int G,
                const int32_t* __restrict__ iou_arg, const int32_t* __restrict__ cls, const int32_t* __restrict__ list_pos,
                const int32_t* __restrict__ counts, int max_targets, double sd0, double sd1, double sd2, double sd3,
                double* __restrict__ target_bbox, double* __restrict__ positive_anchors) {
  pdl_prologue();
  __shared__ int scratch[33];
  const int b = blockIdx.x, tid = threadIdx.x;
  const int32_t* c = cls + (int64_t)b * A;
  const int32_t* lst = list_pos + (int64_t)b * A;
  const int n_pos0 = counts[(int64_t)b * 4];
  double* tb = target_bbox + (int64_t)b * max_targets * 4;
  double* pa = positive_anchors + (int64_t)b * max_targets * 4;
  for (int i = tid; i < max_targets * 4; i += kRpnSubThreads) {
    tb[i] = 0.0;
    pa[i] = 0.0;
  }
  __syncthreads();
  cta_compact(n_pos0, [&](int r0) { return c[lst[r0]] == 1; },
               [&](int r0, int r) {
                 if (r >= max_targets) return;
                 const int i = lst[r0];
                 const double* an = anchors + 4 * (int64_t)i;
                 const double* g = gt + ((int64_t)b * G + iou_arg[(int64_t)b * A + i]) * 4;
                 const double ah = an[2] - an[0], aw = an[3] - an[1];
                 const double acy = an[0] + 0.5 * ah, acx = an[1] + 0.5 * aw;
                 const double gh = g[2] - g[0], gw = g[3] - g[1];
                 const double gcy = g[0] + 0.5 * gh, gcx = g[1] + 0.5 * gw;
                 tb[r * 4 + 0] = ((gcy - acy) / ah) / sd0;
                 tb[r * 4 + 1] = ((gcx - acx) / aw) / sd1;
                 tb[r * 4 + 2] = log(gh / ah) / sd2;
                 tb[r * 4 + 3] = log(gw / aw) / sd3;
                 pa[r * 4 + 0] = an[0]; pa[r * 4 + 1] = an[1]; pa[r * 4 + 2] = an[2]; pa[r * 4 + 3] = an[3];
               },
               scratch);
}

}  // namespace od

using namespace od;

extern "C" {

struct RpnWs {
  double* iou_max;
  int32_t* iou_arg;
  int32_t* list_pos;
  int32_t* list_neg;
  int32_t* gt_best;
  float4* anchors_c;
  int2* cnt;
  int2* pcnt;
  double* part_v;
  int32_t* part_i;
};
static size_t carve_rpn_ws(Workspace& w, int64_t B, int64_t A, int64_t G, RpnWs* out) {
  RpnWs r;
  const int64_t g1 = G > 0 ? G : 1;
  const int64_t nchunk = (A + kChunk - 1) / kChunk, nblk = (A + kRpnThreads - 1) / kRpnThreads;
  r.iou_max = w.take<double>((size_t)(B * A));
  r.iou_arg = w.take<int32_t>((size_t)(B * A));
  r.list_pos = w.take<int32_t>((size_t)(B * A));
  r.list_neg = w.take<int32_t>((size_t)(B * A));
  r.gt_best = w.take<int32_t>((size_t)(B * g1));
  r.anchors_c = w.take<float4>((size_t)A);
  r.cnt = w.take<int2>((size_t)(B * nchunk));
  r.pcnt = w.take<int2>((size_t)(B * nchunk));
  const bool fused = G > 0 && G <= kFusedMaxGt;
  r.part_v = w.take<double>((size_t)(fused ? B * G * nblk : 1));
  r.part_i = w.take<int32_t>((size_t)(fused ? B * G * nblk : 1));
  if (out) *out = r;
  return w.off + 256;
}

size_t od_rpn_target_workspace_bytes(int64_t batch, int64_t num_anchors, int64_t num_gt) {
  Workspace w(nullptr, 0);
  return carve_rpn_ws(w, batch, num_anchors, num_gt, nullptr);
}

int od_rpn_target_forward(const DLTensor* anchors, const DLTensor* gt_boxes, const DLTensor* gt_count,
                          const DLTensor* perm_pos, const DLTensor* perm_neg, const od_rpn_target_params* params,
                          DLTensor* rpn_target_class, DLTensor* rpn_target_bbox, DLTensor* positive_anchors,
                          DLTensor* counts, void* ws, size_t ws_bytes, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (!params) OD_FAIL(OD_ERR_NULL, "params is NULL");
  DeviceScope scope;
  OD_CHECK(check_tensor(anchors, "anchors", F64, {kAny, 4}, 8, scope));
  OD_CHECK(check_tensor(gt_boxes, "gt_boxes", F64, {kAny, kAny, 4}, 8, scope));
  const int64_t A = anchors->shape[0], B = gt_boxes->shape[0], G = gt_boxes->shape[1], T = params->max_rpn_targets;
  OD_CHECK(check_tensor(gt_count, "gt_count", I32, {B}, 4, scope));
  OD_CHECK(check_tensor(perm_pos, "perm_pos", I32, {B, A}, 4, scope));
  OD_CHECK(check_tensor(perm_neg, "perm_neg", I32, {B, A}, 4, scope));
  OD_CHECK(check_tensor(rpn_target_class, "rpn_target_class", I32, {B, A}, 4, scope));
  OD_CHECK(check_tensor(rpn_target_bbox, "rpn_target_bbox", F64, {B, T, 4}, 8, scope));
  OD_CHECK(check_tensor(positive_anchors, "positive_anchors", F64, {B, T, 4}, 8, scope));
  OD_CHECK(check_tensor(counts, "counts", I32, {B, 4}, 4, scope));
  if (A >= (1ll << 30) || G > 4096 || B > 65535) OD_FAIL(OD_ERR_PARAM, "supports A < 2^30, G <= 4096, B <= 65535");
  if (B == 0 || A == 0) return OD_OK;
  if (!ws) OD_FAIL(OD_ERR_WORKSPACE, "workspace is NULL");
  Workspace w(ws, ws_bytes);
  RpnWs r;
  carve_rpn_ws(w, B, A, G, &r);
  if (!w.ok()) OD_FAIL(OD_ERR_WORKSPACE, "workspace %zu < %zu bytes", ws_bytes, w.off);
  const double* an = dptr<double>(anchors);
  const double* gt = dptr<double>(gt_boxes);
  const int32_t* gc = dptr<int32_t>(gt_count);
  int32_t* cls = dptr<int32_t>(rpn_target_class);
  const int64_t g1 = G > 0 ? G : 1;
  const bool fused = G > 0 && G <= kFusedMaxGt;
  {
    const dim3 grid((unsigned)((A + kRpnThreads - 1) / kRpnThreads), (unsigned)B);
    size_t smem = ((size_t)g1 * 5 + 1) * sizeof(double) + (size_t)g1 * sizeof(float4);
    if (fused) {
      smem += (size_t)kRpnWarps * G * (sizeof(double) + sizeof(int32_t));
      OD_CUDA(launch_pdl(rpn_anchor_best_kernel<true>, grid, dim3(kRpnThreads), smem, st, an, (int)A, gt, gc, (int)G, r.iou_max, r.iou_arg, r.anchors_c,
                                                                     r.part_v, r.part_i));
    } else {
      static const size_t best_static = static_smem_bytes((const void*)rpn_anchor_best_kernel<false>);
      if (smem + best_static > 48 * 1024)
        OD_CUDA(cudaFuncSetAttribute(rpn_anchor_best_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      OD_CUDA(launch_pdl(rpn_anchor_best_kernel<false>, grid, dim3(kRpnThreads), smem, st, an, (int)A, gt, gc, (int)G, r.iou_max, r.iou_arg, r.anchors_c,
                                                                      nullptr, nullptr));
    }
    OD_LAUNCH_CHECK("rpn_anchor_best_kernel");
    if (fused) {
      OD_CUDA(launch_pdl(rpn_gt_reduce_kernel, dim3((unsigned)G, (unsigned)B), dim3(kRpnThreads), 0, st, r.part_v, r.part_i, (int)grid.x, gc, (int)G, r.gt_best));
      OD_LAUNCH_CHECK("rpn_gt_reduce_kernel");
    } else if (G > 0) {
      OD_CUDA(launch_pdl(rpn_gt_best_kernel, dim3((unsigned)G, (unsigned)B), dim3(kRpnThreads), 0, st, an, r.anchors_c, (int)A, gt, gc, (int)G, r.gt_best));
      OD_LAUNCH_CHECK("rpn_gt_best_kernel");
    }
  }
  {
    const int64_t total = B * A;
    OD_CUDA(launch_pdl(rpn_label_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, st, r.iou_max, total, cls));
    OD_LAUNCH_CHECK("rpn_label_kernel");
  }
  if (G > 0) {
    const dim3 grid((unsigned)((G + 127) / 128), (unsigned)B);
    OD_CUDA(launch_pdl(rpn_label_best_kernel, grid, dim3(128), 0, st, r.gt_best, (int)G, (int)A, cls));
    OD_LAUNCH_CHECK("rpn_label_best_kernel");
  }
  {
    const dim3 grid((unsigned)((A + kChunk - 1) / kChunk), (unsigned)B);
    const int32_t* pp = dptr<int32_t>(perm_pos);
    const int32_t* pn = dptr<int32_t>(perm_neg);
    int32_t* cnts = dptr<int32_t>(counts);
    OD_CUDA(launch_pdl(rpn_count_kernel, grid, dim3(kRpnThreads), 0, st, cls, (int)A, r.cnt));
    OD_LAUNCH_CHECK("rpn_count_kernel");
    OD_CUDA(launch_pdl(rpn_compact_kernel, grid, dim3(kRpnThreads), 0, st, cls, (int)A, r.cnt, (int)T, r.list_pos, r.list_neg, cnts));
    OD_LAUNCH_CHECK("rpn_compact_kernel");
    OD_CUDA(launch_pdl(rpn_perm_kernel<false>, grid, dim3(kRpnThreads), 0, st, pp, pn, (int)A, r.cnt, r.pcnt, (int)T, r.list_pos, r.list_neg, cls));
    OD_LAUNCH_CHECK("rpn_perm_kernel<count>");
    OD_CUDA(launch_pdl(rpn_perm_kernel<true>, grid, dim3(kRpnThreads), 0, st, pp, pn, (int)A, r.cnt, r.pcnt, (int)T, r.list_pos, r.list_neg, cls));
    OD_LAUNCH_CHECK("rpn_perm_kernel<apply>");
    OD_CUDA(launch_pdl(rpn_emit_kernel, dim3((unsigned)B), dim3(kRpnSubThreads), 0, st, an, (int)A, gt, (int)G, r.iou_arg, cls, r.list_pos, cnts, (int)T,
                                                            params->bbox_stddev[0], params->bbox_stddev[1], params->bbox_stddev[2],
                                                            params->bbox_stddev[3], dptr<double>(rpn_target_bbox),
                                                            dptr<double>(positive_anchors)));
    OD_LAUNCH_CHECK("rpn_emit_kernel");
  }
  return OD_OK;
}

}  // extern "C"
