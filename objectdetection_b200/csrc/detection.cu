// detection.cu — DetectionLayer.build (detection.py:80-260):
//   argmax class -> class-specific delta decode -> clip to the normalised window -> fg & score filter
//   -> per-class NMS -> top-M by (score desc, ROI index asc) -> rows (y1,x1,y2,x2,class,score), zero padded.
//
// Per-class NMS is one class-segmented bitmask NMS: kept ROIs are ordered by (class, score desc, index asc)
// with a 64-bit key sort, the IoU bitmask only links boxes of the same class (nms.cu `group`), one scan
// resolves all classes, and the per-class cap of M (max_output_size of each tf.image.non_max_suppression
// call, detection.py:177-182) is applied afterwards from a prefix count inside each class segment — boxes
// beyond the cap are the lowest ranked of their class and can only suppress boxes that are dropped anyway.
#include "nms.cuh"
#include "topk.cuh"

namespace od {

constexpr int kFinThreads = 1024;

struct DetDebugPtrs {
  int32_t* class_ids;
  float* class_scores;
  float4* bbox_delta;
  float4* refined;
  float4* clipped;
  int32_t* keep_mask;
};

// One warp per ROI slot (slots >= N only clear their sort key). TP, TB: the dtypes (float or bf16) of the probabilities
// and of the box deltas; bf16 values are widened exactly, so the scan and the decode are the fp32 ones on those values.
template <typename TP, typename TB>
__device__ __forceinline__ void det_prepare_body(const float4* __restrict__ proposals, const TP* __restrict__ probs,
                                                 const TB* __restrict__ bbox, const float4* __restrict__ window, int N,
                                                 int C, int n_pow2, float4 stddev, float min_conf,
                                                 int32_t* __restrict__ cls_out, float* __restrict__ score_out,
                                                 float4* __restrict__ clipped_out, unsigned long long* __restrict__ keys,
                                                 int32_t* __restrict__ num_valid, const DetDebugPtrs& dbg) {
  const int lane = threadIdx.x & 31;
  const int64_t slot = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int b = blockIdx.y;
  if (slot >= n_pow2) return;
  if (slot >= N) {
    if (lane == 0) keys[(int64_t)b * n_pow2 + slot] = 0ull;
    return;
  }
  if (slot == 0 && lane == 0) num_valid[b] = 0;   // det_rank_gather_kernel raises it with atomicMax
  const int n = (int)slot;
  const int64_t r = (int64_t)b * N + n;
  const TP* p = probs + r * C;
  // argmax, first maximum (detection.py:115), as the sequential `best = p[0]; if (p[c] > best)` scan decides it: a NaN
  // in p[0] wins (nothing compares greater), a NaN anywhere else is never taken. A lane's own first value is the only
  // one it takes without a compare, so lanes other than 0 drop a NaN there.
  float best = -INFINITY;
  int arg = 0x7fffffff;
  if (lane < C) {
    best = ld_head(p + lane);
    arg = lane;
    if (lane > 0 && best != best) {
      best = -INFINITY;
      arg = 0x7fffffff;
    }
    for (int c = lane + 32; c < C; c += 32) {
      const float v = ld_head(p + c);
      if (v > best) {
        best = v;
        arg = c;
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, best, o);
    const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
    if (ov > best || (ov == best && oa < arg)) {
      best = ov;
      arg = oa;
    }
  }
  if (lane != 0) return;
  if (arg == 0x7fffffff) arg = 0;
  const float score = ld_head(p + arg);                                              // :129
  const float4 raw = ldg_head4(bbox, r * C + arg);
  const float4 d = make_float4(raw.x * stddev.x, raw.y * stddev.y, raw.z * stddev.z, raw.w * stddev.w);  // :117,:130
  const float4 ref = decode_box(proposals[r], d);                                    // :133
  const float4 cl = clip_box(ref, window[b]);                                        // :147
  const bool keep = (arg > 0) && (score > min_conf);                                 // :152-158
  cls_out[r] = arg;
  score_out[r] = score;
  clipped_out[r] = cl;
  keys[(int64_t)b * n_pow2 + n] =
      keep ? (((unsigned long long)(C - arg) << 48) | ((unsigned long long)score_key(score) << 16) |
              (unsigned long long)(0xFFFFu - (uint32_t)n))
           : (unsigned long long)(0xFFFFu - (uint32_t)n);   // dropped ROIs: class field 0, still unique (rank sort)
  if (dbg.class_ids) dbg.class_ids[r] = arg;
  if (dbg.class_scores) dbg.class_scores[r] = score;
  if (dbg.bbox_delta) dbg.bbox_delta[r] = d;
  if (dbg.refined) dbg.refined[r] = ref;
  if (dbg.clipped) dbg.clipped[r] = cl;
  if (dbg.keep_mask) dbg.keep_mask[r] = keep ? 1 : 0;
}
__global__ void __launch_bounds__(256)
det_prepare_kernel(const float4* __restrict__ proposals, const float* __restrict__ probs,
                   const float4* __restrict__ bbox, const float4* __restrict__ window, int N, int C, int n_pow2,
                   float4 stddev, float min_conf, int32_t* __restrict__ cls_out, float* __restrict__ score_out,
                   float4* __restrict__ clipped_out, unsigned long long* __restrict__ keys,
                   int32_t* __restrict__ num_valid, DetDebugPtrs dbg) {
  det_prepare_body<float, float>(proposals, probs, reinterpret_cast<const float*>(bbox), window, N, C, n_pow2, stddev,
                                 min_conf, cls_out, score_out, clipped_out, keys, num_valid, dbg);
}
// bf16 probabilities and / or box deltas: the same body, an overload of the same name (the fp32 kernel above keeps its
// name)
template <typename TP, typename TB>
__global__ void __launch_bounds__(256)
det_prepare_kernel(const float4* __restrict__ proposals, const TP* __restrict__ probs, const TB* __restrict__ bbox,
                   const float4* __restrict__ window, int N, int C, int n_pow2, float4 stddev, float min_conf,
                   int32_t* __restrict__ cls_out, float* __restrict__ score_out, float4* __restrict__ clipped_out,
                   unsigned long long* __restrict__ keys, int32_t* __restrict__ num_valid, DetDebugPtrs dbg) {
  det_prepare_body<TP, TB>(proposals, probs, bbox, window, N, C, n_pow2, stddev, min_conf, cls_out, score_out,
                           clipped_out, keys, num_valid, dbg);
}

// Rank sort of the N keys of one image fused with the gather: keys are unique, the sorted position of a key is the
// number of keys greater than it. grid (ceil(N/64), B); a CTA owns 64 keys, its 4 thread groups each count over a
// quarter of every 1024-key tile in shared memory. Writes the sorted key, box and class of position `rank`, and
// num_valid = number of kept ROIs (keys whose class field is non-zero sort first).
constexpr int kDetRankThreads = 256;
constexpr int kDetRankMine = 64;
constexpr int kDetRankTile = 1024;
__global__ void __launch_bounds__(kDetRankThreads)
det_rank_gather_kernel(const unsigned long long* __restrict__ keys, const float4* __restrict__ clipped,
                       const int32_t* __restrict__ cls, int N, int n_pow2, unsigned long long* __restrict__ sorted_keys,
                       float4* __restrict__ sorted_boxes, int32_t* __restrict__ group, int32_t* __restrict__ num_valid) {
  __shared__ unsigned long long tile[kDetRankTile];
  __shared__ int32_t partial[kDetRankThreads];
  const int b = blockIdx.y;
  const unsigned long long* in = keys + (int64_t)b * n_pow2;
  const int me = blockIdx.x * kDetRankMine + (threadIdx.x & (kDetRankMine - 1));
  const int part = threadIdx.x / kDetRankMine;
  constexpr int kParts = kDetRankThreads / kDetRankMine;
  const unsigned long long mine = (me < N) ? in[me] : ~0ull;
  int rank = 0;
  for (int t0 = 0; t0 < N; t0 += kDetRankTile) {
    __syncthreads();
    for (int i = threadIdx.x; i < kDetRankTile; i += kDetRankThreads) tile[i] = (t0 + i < N) ? in[t0 + i] : 0ull;
    __syncthreads();
    const unsigned long long* tp = tile + part * (kDetRankTile / kParts);
#pragma unroll 16
    for (int j = 0; j < kDetRankTile / kParts; ++j) rank += (tp[j] > mine) ? 1 : 0;
  }
  partial[threadIdx.x] = rank;
  __syncthreads();
  if (part == 0 && me < N) {
#pragma unroll
    for (int q = 1; q < kParts; ++q) rank += partial[threadIdx.x + q * kDetRankMine];
    const bool valid = (mine >> 48) != 0ull;
    const int n = (int)(0xFFFFu - (uint32_t)(mine & 0xFFFFull));
    OD_DBG_IDX(rank, N);
    sorted_keys[(int64_t)b * n_pow2 + rank] = valid ? mine : 0ull;
    sorted_boxes[(int64_t)b * N + rank] = valid ? clipped[(int64_t)b * N + n] : make_float4(0.f, 0.f, 0.f, 0.f);
    group[(int64_t)b * N + rank] = valid ? cls[(int64_t)b * N + n] : -1;
    if (valid) atomicMax(&num_valid[b], rank + 1);
  }
}

// Sorted position -> box / class; also finds num_valid (keys are sorted descending, zeros last).
__global__ void det_gather_kernel(const unsigned long long* __restrict__ keys, const float4* __restrict__ clipped,
                                  const int32_t* __restrict__ cls, int N, int n_pow2, float4* __restrict__ sorted_boxes,
                                  int32_t* __restrict__ group, int32_t* __restrict__ num_valid) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int b = blockIdx.y;
  if (i >= N) return;
  // kept ROIs carry a non-zero class field and sort first
  const unsigned long long k = keys[(int64_t)b * n_pow2 + i];
  const unsigned long long nxt = (i + 1 < n_pow2) ? keys[(int64_t)b * n_pow2 + i + 1] : 0ull;
  const bool valid = (k >> 48) != 0ull, next_valid = (nxt >> 48) != 0ull;
  if (valid && (!next_valid || i == N - 1)) num_valid[b] = i + 1;   // (num_valid was reset to 0 by det_prepare_kernel)
  if (valid) {
    const int n = (int)(0xFFFFu - (uint32_t)(k & 0xFFFFull));
    sorted_boxes[(int64_t)b * N + i] = clipped[(int64_t)b * N + n];
    group[(int64_t)b * N + i] = cls[(int64_t)b * N + n];
  } else {
    sorted_boxes[(int64_t)b * N + i] = make_float4(0.f, 0.f, 0.f, 0.f);
    group[(int64_t)b * N + i] = -1;
  }
}

// One CTA per image: per-class cap, final top-M ordering, output rows.
__global__ void __launch_bounds__(kFinThreads)
det_finalize_kernel(const unsigned long long* __restrict__ keys, const int32_t* __restrict__ keep_flag,
                    const int32_t* __restrict__ group, const int32_t* __restrict__ num_valid,
                    const float4* __restrict__ clipped, const int32_t* __restrict__ cls,
                    const float* __restrict__ score, int N, int n_pow2, int M, float* __restrict__ detections,
                    int32_t* __restrict__ nms_keep_mask) {
  extern __shared__ unsigned long long fkeys[];                 // [n_pow2]
  int32_t* prefix = reinterpret_cast<int32_t*>(fkeys + n_pow2);  // [n_pow2] inclusive kept count
  __shared__ int32_t warp_sums[kFinThreads / 32];
  __shared__ int32_t tile_base;
  const int b = blockIdx.x;
  const int nv = num_valid[b];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int32_t* kf = keep_flag + (int64_t)b * N;
  const int32_t* grp = group + (int64_t)b * N;
  const unsigned long long* kin = keys + (int64_t)b * n_pow2;
  if (tid == 0) tile_base = 0;
  if (nms_keep_mask)
    for (int n = tid; n < N; n += kFinThreads) nms_keep_mask[(int64_t)b * N + n] = 0;
  __syncthreads();
  // inclusive prefix count of kept flags over sorted positions
  for (int t0 = 0; t0 < nv; t0 += kFinThreads) {
    const int i = t0 + tid;
    const int f = (i < nv) ? kf[i] : 0;
    int incl = f;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += v;
    }
    if (lane == 31) warp_sums[warp] = incl;
    __syncthreads();
    int off = tile_base;
    for (int w = 0; w < warp; ++w) off += warp_sums[w];
    if (i < nv) prefix[i] = off + incl;
    __syncthreads();
    if (tid == kFinThreads - 1) tile_base = off + incl;
    __syncthreads();
  }
  // survivors of the per-class cap -> final ordering key (score desc, ROI index asc), compacted into fkeys[0..m)
  int32_t m = 0;
  for (int t0 = 0; t0 < nv; t0 += kFinThreads) {
    const int i = t0 + tid;
    unsigned long long out = 0ull;
    if (i < nv && kf[i]) {
      const int g = grp[i];
      int lo = 0, hi = i;  // first position of this class segment (classes ascend along sorted positions)
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (grp[mid] < g) lo = mid + 1;
        else hi = mid;
      }
      const int before = (lo > 0) ? prefix[lo - 1] : 0;
      const int rank = prefix[i] - 1 - before;  // kept boxes of this class ahead of i
      if (rank < M) {
        const unsigned long long k = kin[i];
        const uint32_t n = 0xFFFFu - (uint32_t)(k & 0xFFFFull);
        const uint32_t skey = (uint32_t)((k >> 16) & 0xFFFFFFFFull);
        out = ((unsigned long long)skey << 32) | (unsigned long long)(0xFFFFFFFFu - n);
        OD_DBG_IDX(n, N);
        if (nms_keep_mask) nms_keep_mask[(int64_t)b * N + n] = 1;
      }
    }
    // stable block compaction of the non-zero keys
    const uint32_t bal = __ballot_sync(0xffffffffu, out != 0ull);
    if (lane == 0) warp_sums[warp] = __popc(bal);
    __syncthreads();
    int off = m, total = 0;
    for (int w = 0; w < kFinThreads / 32; ++w) {
      const int c = warp_sums[w];
      if (w < warp) off += c;
      total += c;
    }
    if (out != 0ull) {
      OD_DBG_IDX(off + __popc(bal & ((1u << lane) - 1u)), n_pow2);
      fkeys[off + __popc(bal & ((1u << lane) - 1u))] = out;
    }
    m += total;
    __syncthreads();
  }
  // rank of every survivor among the m survivors (keys are unique) = its output row; rows >= min(m, M) stay zero
  float* det = detections + (int64_t)b * M * 6;
  for (int t = tid; t < m; t += kFinThreads) {
    const unsigned long long mine = fkeys[t];
    int rank = 0;
    for (int j = 0; j < m; ++j) rank += (fkeys[j] > mine) ? 1 : 0;
    if (rank < M) {
      const int n = (int)composite_index(mine);
      const float4 bx = clipped[(int64_t)b * N + n];
      float* row = det + (int64_t)rank * 6;
      row[0] = bx.x; row[1] = bx.y; row[2] = bx.z; row[3] = bx.w;
      OD_DBG_IDX(n, N);
      row[4] = (float)cls[(int64_t)b * N + n];
      row[5] = score[(int64_t)b * N + n];
    }
  }
  for (int j = min(m, M) + tid; j < M; j += kFinThreads) {
#pragma unroll
    for (int c = 0; c < 6; ++c) det[j * 6 + c] = 0.0f;
  }
}

// unmold_detection (detection.py:8-53) + denorm_boxes (utils.py:212-227) for a whole batch on the device (SURVEY.md
// §8f rank 2: the step after the path, e.g. straight after the all-gather). One CTA per image:
//   N = first row with class_id == 0; boxes = (boxes - shift) / scale in fp32 (window frame), then
//   around(boxes * (h-1, w-1, h-1, w-1) + (0,0,1,1)) in fp64 -> int32 (numpy promotes float32 * int64 to float64;
//   around = half to even); rows with (y2-y1)*(x2-x1) <= 0 are dropped; survivors keep their order.
constexpr int kUnmoldThreads = 128;
__global__ void __launch_bounds__(kUnmoldThreads)
unmold_kernel(const float* __restrict__ detections, const float4* __restrict__ window_norm,
              const int32_t* __restrict__ original_shape, int M, int32_t* __restrict__ boxes, int32_t* __restrict__ class_ids,
              float* __restrict__ scores, int32_t* __restrict__ counts) {
  __shared__ int s_first_zero;
  __shared__ int warp_cnt[kUnmoldThreads / 32];
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float* det = detections + (int64_t)b * M * 6;
  if (tid == 0) s_first_zero = M;
  __syncthreads();
  for (int i = tid; i < M; i += kUnmoldThreads)
    if (det[i * 6 + 4] == 0.0f) atomicMin(&s_first_zero, i);
  __syncthreads();
  const int N = s_first_zero;
  const float4 w = window_norm[b];
  const float wh = w.z - w.x, ww = w.w - w.y;
  const double sh = (double)(original_shape[b * 2 + 0] - 1), sw = (double)(original_shape[b * 2 + 1] - 1);
  int32_t* ob = boxes + (int64_t)b * M * 4;
  int32_t* oc = class_ids + (int64_t)b * M;
  float* os = scores + (int64_t)b * M;
  int base = 0;
  for (int t0 = 0; t0 < N; t0 += kUnmoldThreads) {
    const int i = t0 + tid;
    bool keep = false;
    int y1 = 0, x1 = 0, y2 = 0, x2 = 0;
    if (i < N) {
      const float by1 = (det[i * 6 + 0] - w.x) / wh, bx1 = (det[i * 6 + 1] - w.y) / ww;
      const float by2 = (det[i * 6 + 2] - w.x) / wh, bx2 = (det[i * 6 + 3] - w.y) / ww;
      y1 = (int)rint((double)by1 * sh + 0.0);
      x1 = (int)rint((double)bx1 * sw + 0.0);
      y2 = (int)rint((double)by2 * sh + 1.0);
      x2 = (int)rint((double)bx2 * sw + 1.0);
      keep = (y2 - y1) * (x2 - x1) > 0;
    }
    const uint32_t bal = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) warp_cnt[warp] = __popc(bal);
    __syncthreads();
    int off = base, total = 0;
    for (int q = 0; q < kUnmoldThreads / 32; ++q) {
      if (q < warp) off += warp_cnt[q];
      total += warp_cnt[q];
    }
    if (keep) {
      const int r = off + __popc(bal & ((1u << lane) - 1u));
      ob[r * 4 + 0] = y1; ob[r * 4 + 1] = x1; ob[r * 4 + 2] = y2; ob[r * 4 + 3] = x2;
      oc[r] = (int32_t)det[i * 6 + 4];
      os[r] = det[i * 6 + 5];
    }
    base += total;
    __syncthreads();
  }
  for (int r = base + tid; r < M; r += kUnmoldThreads) {
    ob[r * 4 + 0] = 0; ob[r * 4 + 1] = 0; ob[r * 4 + 2] = 0; ob[r * 4 + 3] = 0;
    oc[r] = 0;
    os[r] = 0.0f;
  }
  if (tid == 0) counts[b] = base;
}

struct DetWs {
  int32_t* cls;
  float* score;
  float4* clipped;
  unsigned long long* keys;
  unsigned long long* sorted_keys;
  float4* sorted_boxes;
  int32_t* group;
  int32_t* num_valid;
  int32_t* keep_flag;
  void* nms_ws;
  size_t nms_bytes;
};
static size_t carve_det_ws(Workspace& w, int64_t B, int64_t N, DetWs* out) {
  DetWs d;
  const int64_t n_pow2 = next_pow2(N > 0 ? N : 1);
  d.cls = w.take<int32_t>((size_t)(B * N));
  d.score = w.take<float>((size_t)(B * N));
  d.clipped = w.take<float4>((size_t)(B * N));
  d.keys = w.take<unsigned long long>((size_t)(B * n_pow2));
  d.sorted_keys = w.take<unsigned long long>((size_t)(B * n_pow2));
  d.sorted_boxes = w.take<float4>((size_t)(B * N));
  d.group = w.take<int32_t>((size_t)(B * N));
  d.num_valid = w.take<int32_t>((size_t)B);
  d.keep_flag = w.take<int32_t>((size_t)(B * N));
  d.nms_bytes = nms_sorted_workspace_bytes(B, N);
  d.nms_ws = w.take<char>(d.nms_bytes);
  if (out) *out = d;
  return w.off + 256;
}

}  // namespace od

using namespace od;

extern "C" {

size_t od_detection_workspace_bytes(int64_t batch, int64_t num_rois, int64_t num_classes) {
  Workspace w(nullptr, 0);
  return carve_det_ws(w, batch, num_rois, nullptr);
}

int od_detection_forward(const DLTensor* proposals, const DLTensor* mrcnn_class_probs, const DLTensor* mrcnn_bbox,
                         const DLTensor* window_norm, const od_detection_params* params, DLTensor* detections,
                         const od_detection_debug* debug, void* ws, size_t ws_bytes, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (!params) OD_FAIL(OD_ERR_NULL, "params is NULL");
  DeviceScope scope;
  OD_CHECK(check_tensor(proposals, "proposals", F32, {kAny, kAny, 4}, 16, scope));
  const DType probs_dt = f32_or_bf16(mrcnn_class_probs), bbox_dt = f32_or_bf16(mrcnn_bbox);
  OD_CHECK(check_tensor(mrcnn_class_probs, "mrcnn_class_probs", probs_dt, {proposals->shape[0], proposals->shape[1], kAny},
                        probs_dt == BF16 ? 2 : 4, scope));
  const int64_t B = mrcnn_class_probs->shape[0], N = mrcnn_class_probs->shape[1], C = mrcnn_class_probs->shape[2];
  const int64_t M = params->max_instances;
  OD_CHECK(check_tensor(mrcnn_bbox, "mrcnn_bbox", bbox_dt, {B, N, C, 4}, bbox_dt == BF16 ? 8 : 16, scope));
  OD_CHECK(check_tensor(window_norm, "window_norm", F32, {B, 4}, 16, scope));
  OD_CHECK(check_tensor(detections, "detections", F32, {B, M, 6}, 4, scope));
  if (N > 16384 || C > 65535 || C < 1) OD_FAIL(OD_ERR_PARAM, "DetectionLayer supports N <= 16384 ROIs and 1 <= C <= 65535 classes");
  if (B > 65535) OD_FAIL(OD_ERR_PARAM, "batch > 65535");
  od_detection_debug dbg;
  memset(&dbg, 0, sizeof(dbg));
  if (debug) dbg = *debug;
  OD_CHECK(check_opt_tensor(dbg.class_ids, "debug.class_ids", I32, {B, N}, 4, scope));
  OD_CHECK(check_opt_tensor(dbg.class_scores, "debug.class_scores", F32, {B, N}, 4, scope));
  OD_CHECK(check_opt_tensor(dbg.bbox_delta, "debug.bbox_delta", F32, {B, N, 4}, 16, scope));
  OD_CHECK(check_opt_tensor(dbg.refined_proposals, "debug.refined_proposals", F32, {B, N, 4}, 16, scope));
  OD_CHECK(check_opt_tensor(dbg.clipped_proposals, "debug.clipped_proposals", F32, {B, N, 4}, 16, scope));
  OD_CHECK(check_opt_tensor(dbg.keep_mask, "debug.keep_mask", I32, {B, N}, 4, scope));
  OD_CHECK(check_opt_tensor(dbg.nms_keep_mask, "debug.nms_keep_mask", I32, {B, N}, 4, scope));
  if (B == 0 || M == 0) return OD_OK;
  if (N == 0) {
    OD_CUDA(cudaMemsetAsync(dptr<float>(detections), 0, sizeof(float) * (size_t)(B * M * 6), st));
    return OD_OK;
  }
  if (!ws) OD_FAIL(OD_ERR_WORKSPACE, "workspace is NULL");
  Workspace w(ws, ws_bytes);
  DetWs d;
  carve_det_ws(w, B, N, &d);
  if (!w.ok()) OD_FAIL(OD_ERR_WORKSPACE, "workspace %zu < %zu bytes", ws_bytes, w.off);
  const int n_pow2 = (int)next_pow2(N);
  const float4 sd = make_float4(params->bbox_stddev[0], params->bbox_stddev[1], params->bbox_stddev[2], params->bbox_stddev[3]);
  DetDebugPtrs dp;
  dp.class_ids = dptr<int32_t>(dbg.class_ids);
  dp.class_scores = dptr<float>(dbg.class_scores);
  dp.bbox_delta = dptr<float4>(dbg.bbox_delta);
  dp.refined = dptr<float4>(dbg.refined_proposals);
  dp.clipped = dptr<float4>(dbg.clipped_proposals);
  dp.keep_mask = dptr<int32_t>(dbg.keep_mask);
  {
    const dim3 grid((unsigned)(((int64_t)n_pow2 * 32 + 255) / 256), (unsigned)B);
    using BF = __nv_bfloat16;
    const float4* pr = dptr<float4>(proposals);
    const float4* win = dptr<float4>(window_norm);
    const float mc = params->min_confidence;
    if (probs_dt == BF16 && bbox_dt == BF16)
      det_prepare_kernel<BF, BF><<<grid, 256, 0, st>>>(pr, dptr<BF>(mrcnn_class_probs), dptr<BF>(mrcnn_bbox), win, (int)N,
                                                       (int)C, n_pow2, sd, mc, d.cls, d.score, d.clipped, d.keys, d.num_valid, dp);
    else if (probs_dt == BF16)
      det_prepare_kernel<BF, float><<<grid, 256, 0, st>>>(pr, dptr<BF>(mrcnn_class_probs), dptr<float>(mrcnn_bbox), win,
                                                          (int)N, (int)C, n_pow2, sd, mc, d.cls, d.score, d.clipped, d.keys,
                                                          d.num_valid, dp);
    else if (bbox_dt == BF16)
      det_prepare_kernel<float, BF><<<grid, 256, 0, st>>>(pr, dptr<float>(mrcnn_class_probs), dptr<BF>(mrcnn_bbox), win,
                                                          (int)N, (int)C, n_pow2, sd, mc, d.cls, d.score, d.clipped, d.keys,
                                                          d.num_valid, dp);
    else
      det_prepare_kernel<<<grid, 256, 0, st>>>(pr, dptr<float>(mrcnn_class_probs), dptr<float4>(mrcnn_bbox), win, (int)N,
                                               (int)C, n_pow2, sd, mc, d.cls, d.score, d.clipped, d.keys, d.num_valid, dp);
    OD_LAUNCH_CHECK("det_prepare_kernel");
  }
  const unsigned long long* sorted_keys = d.sorted_keys;
  if (N <= 4096) {
    const dim3 grid((unsigned)((N + kDetRankMine - 1) / kDetRankMine), (unsigned)B);
    det_rank_gather_kernel<<<grid, kDetRankThreads, 0, st>>>(d.keys, d.clipped, d.cls, (int)N, n_pow2, d.sorted_keys,
                                                            d.sorted_boxes, d.group, d.num_valid);
    OD_LAUNCH_CHECK("det_rank_gather_kernel");
  } else {   // many ROIs: bitonic sort in place, then gather
    OD_CHECK(sort_u64_desc_launch(d.keys, B, n_pow2, st));
    const dim3 grid((unsigned)((N + 255) / 256), (unsigned)B);
    det_gather_kernel<<<grid, 256, 0, st>>>(d.keys, d.clipped, d.cls, (int)N, n_pow2, d.sorted_boxes, d.group, d.num_valid);
    OD_LAUNCH_CHECK("det_gather_kernel");
    sorted_keys = d.keys;
  }
  OD_CHECK(nms_sorted_launch(d.sorted_boxes, d.num_valid, d.group, B, N, params->nms_threshold, N, nullptr, nullptr,
                             d.keep_flag, d.nms_ws, d.nms_bytes, st));
  {
    const size_t smem = (size_t)n_pow2 * (sizeof(unsigned long long) + sizeof(int32_t));
    OD_CUDA(cudaFuncSetAttribute(det_finalize_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    det_finalize_kernel<<<(unsigned)B, kFinThreads, smem, st>>>(sorted_keys, d.keep_flag, d.group, d.num_valid, d.clipped, d.cls,
                                                                d.score, (int)N, n_pow2, (int)M, dptr<float>(detections),
                                                                dptr<int32_t>(dbg.nms_keep_mask));
    OD_LAUNCH_CHECK("det_finalize_kernel");
  }
  return OD_OK;
}

int od_unmold_detections(const DLTensor* detections, const DLTensor* window_norm, const DLTensor* original_shape,
                         DLTensor* boxes, DLTensor* class_ids, DLTensor* scores, DLTensor* counts, void* stream) {
  DeviceScope scope;
  OD_CHECK(check_tensor(detections, "detections", F32, {kAny, kAny, 6}, 4, scope));
  const int64_t B = detections->shape[0], M = detections->shape[1];
  OD_CHECK(check_tensor(window_norm, "window_norm", F32, {B, 4}, 16, scope));
  OD_CHECK(check_tensor(original_shape, "original_shape", I32, {B, 2}, 4, scope));
  OD_CHECK(check_tensor(boxes, "boxes", I32, {B, M, 4}, 4, scope));
  OD_CHECK(check_tensor(class_ids, "class_ids", I32, {B, M}, 4, scope));
  OD_CHECK(check_tensor(scores, "scores", F32, {B, M}, 4, scope));
  OD_CHECK(check_tensor(counts, "counts", I32, {B}, 4, scope));
  if (B > 0x7FFFFFFFll || M > (1 << 24)) OD_FAIL(OD_ERR_PARAM, "batch / rows out of range");
  if (B == 0) return OD_OK;
  unmold_kernel<<<(unsigned)B, kUnmoldThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      dptr<float>(detections), dptr<float4>(window_norm), dptr<int32_t>(original_shape), (int)M, dptr<int32_t>(boxes),
      dptr<int32_t>(class_ids), dptr<float>(scores), dptr<int32_t>(counts));
  OD_LAUNCH_CHECK("unmold_kernel");
  return OD_OK;
}

}  // extern "C"
