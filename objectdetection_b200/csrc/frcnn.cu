// frcnn.cu — Faster R-CNN single-level proposal layer (FasterRCNN/building_blocks/proposals.py:392-512):
// 9 base anchors + stride-16 shifts -> decode (+1 pixel widths, x1y1x2y2) -> clip -> min-size filter -> top-N by
// score -> greedy NMS (areas (w+1)(h+1), suppress iff ovr >= thr) -> [n,5] rows (b,x1,y1,x2,y2).
// A batch of B images runs as one chain: every kernel takes the image from a grid dimension and works on that image's
// segment of each buffer, so image b's result does not depend on the other images of the batch.
//
// Arithmetic is fp64 like the reference's numpy code (fp32 inputs are widened exactly). The reference's top-N
// (proposals.py:352) argsorts an [n,1] array along its length-1 axis, which selects box 0 n times; this
// implements the intended ranking: flattened (score desc, index asc).
// The IoU bitmask has the same layout as nms.cu's, so the keep scan is shared.
#include "nms.cuh"
#include "topk.cuh"

namespace od {

struct __align__(16) Key128 {
  unsigned long long hi, lo;
};
__device__ __forceinline__ bool key_less(const Key128& a, const Key128& b) {
  return (a.hi < b.hi) || (a.hi == b.hi && a.lo < b.lo);
}
__device__ __forceinline__ unsigned long long d_key(double s) {   // score_key's order: -0 == +0, every NaN above +inf
  if (s != s) return 0xFFFFFFFFFFFFFFFFull;
  s = s + 0.0;
  const unsigned long long b = (unsigned long long)__double_as_longlong(s);
  return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double d_min(double a, double b) { return (b < a) ? b : a; }
__device__ __forceinline__ double d_max(double a, double b) { return (a < b) ? b : a; }

struct FrcnnDev {
  int32_t feat_stride, image_h, image_w, min_box_hw, num_anchors, fw;
  double base[16 * 4];
};

// grid (ceil(total/256), B). Image b reads probs [b] / bbox [b] and writes its segment of boxes [B,total,4], keys
// [B,total] (fp64) or fscore [B,total] (fp32), and its valid counter num_valid[b].
template <typename T>
__global__ void frcnn_decode_kernel(const T* __restrict__ probs, const T* __restrict__ bbox, FrcnnDev p, int64_t total,
                                    double* __restrict__ boxes, Key128* __restrict__ keys, int32_t* __restrict__ num_valid,
                                    float* __restrict__ fscore) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int b = blockIdx.y;
  probs += (int64_t)b * total * 2;   // [h,w,2*na] = 2 * total values per image
  bbox += (int64_t)b * total * 4;
  boxes += (int64_t)b * total * 4;
  Key128 k;
  k.hi = 0ull;                                            // filtered-out rows: below every valid key, still unique
  k.lo = 0xFFFFFFFFFFFFFFFFull - (unsigned long long)i;
  bool valid = false;
  if (i < total) {
    const int na = p.num_anchors;
    const int64_t pos = i / na;
    const int a = (int)(i - pos * na);
    const double sx = (double)((pos % p.fw) * p.feat_stride), sy = (double)((pos / p.fw) * p.feat_stride);
    const double ax1 = p.base[4 * a] + sx, ay1 = p.base[4 * a + 1] + sy;
    const double ax2 = p.base[4 * a + 2] + sx, ay2 = p.base[4 * a + 3] + sy;
    const double dx = (double)bbox[4 * i], dy = (double)bbox[4 * i + 1];
    const double dw = (double)bbox[4 * i + 2], dh = (double)bbox[4 * i + 3];
    // corner_pixels_to_center_inv, proposals.py:286-309
    const double aw = ax2 - ax1 + 1, ah = ay2 - ay1 + 1;
    const double acx = ax1 + aw / 2, acy = ay1 + ah / 2;
    const double pcx = dx * aw + acx, pcy = dy * ah + acy;
    const double pw = exp(dw) * aw, ph = exp(dh) * ah;
    double x1 = pcx - pw / 2, y1 = pcy - ph / 2, x2 = pcx + pw / 2, y2 = pcy + ph / 2;
    // clip_boxes :335-338
    x1 = d_max(d_min(x1, (double)(p.image_w - 1)), 0.0);
    y1 = d_max(d_min(y1, (double)(p.image_h - 1)), 0.0);
    x2 = d_max(d_min(x2, (double)(p.image_w - 1)), 0.0);
    y2 = d_max(d_min(y2, (double)(p.image_h - 1)), 0.0);
    boxes[4 * i] = x1; boxes[4 * i + 1] = y1; boxes[4 * i + 2] = x2; boxes[4 * i + 3] = y2;
    // filter_min_size :342-345
    valid = (x2 - x1 + 1 >= (double)p.min_box_hw) && (y2 - y1 + 1 >= (double)p.min_box_hw);
    if (valid) {
      k.hi = d_key((double)probs[pos * 2 * na + a]);
      k.lo = 0xFFFFFFFFFFFFFFFFull - (unsigned long long)i;
    }
  }
  if (i < total) {
    if (fscore)   // fp32 inputs: the radix-select top-k orders (score desc, index asc) like the 128-bit keys do
      fscore[(int64_t)b * total + i] = valid ? (float)probs[(i / p.num_anchors) * 2 * p.num_anchors + (i % p.num_anchors)] : -INFINITY;
    else
      keys[(int64_t)b * total + i] = k;
  }
  const uint32_t bal = __ballot_sync(0xffffffffu, valid);
  if ((threadIdx.x & 31) == 0 && bal) atomicAdd(&num_valid[b], __popc(bal));
}

// Rank sort fused with the gather: keys are unique, the visiting position of a box is the number of keys of its own
// image greater than its own. grid (ceil(total/32), B); a CTA owns 32 keys of image blockIdx.y, 8 thread groups each
// count over an 8th of every 1024-key tile in shared memory. Position r < K of the image's segment of sorted [B,K,4]
// receives the box (zeros for filtered-out rows); npre[b] = min(num_valid[b], pre_n).
constexpr int kFrRankThreads = 256;
constexpr int kFrRankMine = 32;
constexpr int kFrRankTile = 1024;
__global__ void __launch_bounds__(kFrRankThreads)
frcnn_rank_gather_kernel(const Key128* __restrict__ keys, const double* __restrict__ boxes, int64_t total, int pre_n, int K,
                         double* __restrict__ sorted, const int32_t* __restrict__ num_valid, int32_t* __restrict__ npre) {
  __shared__ unsigned long long tile_hi[kFrRankTile];   // score keys
  __shared__ unsigned long long tile_lo[kFrRankTile];
  __shared__ int32_t partial[kFrRankThreads];
  constexpr int kParts = kFrRankThreads / kFrRankMine;
  const int64_t me = (int64_t)blockIdx.x * kFrRankMine + (threadIdx.x & (kFrRankMine - 1));
  const int part = threadIdx.x / kFrRankMine;
  const int b = blockIdx.y;
  keys += (int64_t)b * total;
  boxes += (int64_t)b * total * 4;
  sorted += (int64_t)b * K * 4;
  if (blockIdx.x == 0 && threadIdx.x == 0) npre[b] = min(num_valid[b], pre_n);
  Key128 mine;
  mine.hi = ~0ull;
  mine.lo = ~0ull;
  if (me < total) mine = keys[me];
  int rank = 0;
  for (int64_t t0 = 0; t0 < total; t0 += kFrRankTile) {
    __syncthreads();
    for (int i = threadIdx.x; i < kFrRankTile; i += kFrRankThreads) {
      Key128 z;
      z.hi = 0ull;
      z.lo = 0ull;
      if (t0 + i < total) z = keys[t0 + i];
      tile_hi[i] = z.hi;
      tile_lo[i] = z.lo;
    }
    __syncthreads();
    const int j0 = part * (kFrRankTile / kParts);
#pragma unroll 8
    for (int j = j0; j < j0 + kFrRankTile / kParts; ++j) {
      const unsigned long long h = tile_hi[j], l = tile_lo[j];   // both loads unconditional: a load behind a branch serialises
      rank += ((h > mine.hi) | ((h == mine.hi) & (l > mine.lo))) ? 1 : 0;
    }
  }
  partial[threadIdx.x] = rank;
  __syncthreads();
  if (part == 0 && me < total) {
#pragma unroll
    for (int q = 1; q < kParts; ++q) rank += partial[threadIdx.x + q * kFrRankMine];
    if (rank < K) {
      const bool valid = mine.hi != 0ull && rank < pre_n;
#pragma unroll
      for (int c = 0; c < 4; ++c) sorted[4 * (int64_t)rank + c] = valid ? boxes[4 * me + c] : 0.0;
    }
  }
}

struct PBox {
  double x1, y1, x2, y2, area;
};
__device__ __forceinline__ PBox load_pbox(const double* b) {
  PBox p;
  p.x1 = b[0]; p.y1 = b[1]; p.x2 = b[2]; p.y2 = b[3];
  p.area = (p.x2 - p.x1 + 1) * (p.y2 - p.y1 + 1);
  return p;
}

// The fp32 screen of frcnn_mask_kernel is exact only while every clipped coordinate is below this bound (see there);
// larger images send every pair to the fp64 path.
constexpr int kFrcnnScreenMaxSide = 8192;

// proposals.py:141-164 as 64x64 tiles (i = kept/earlier box, j = later box). grid (W, W, B): image blockIdx.z reads
// its [K,4] segment of sorted boxes and writes mask [B,K,Ws] and diagT [B,W,64], the layout nms_scan_launch reads.
__global__ void __launch_bounds__(64)
frcnn_mask_kernel(const double* __restrict__ boxes, const int32_t* __restrict__ npre, int K, int W, int Ws, double thr,
                  int screen, unsigned long long* __restrict__ mask, unsigned long long* __restrict__ diagT) {
  const int cb = blockIdx.x, rb = blockIdx.y, b = blockIdx.z;
  if (cb < rb) return;
  const int n = min(npre[b], K);
  if (rb * 64 >= n || cb * 64 >= n) return;
  boxes += (int64_t)b * K * 4;
  mask += (int64_t)b * K * Ws;
  diagT += (int64_t)b * W * 64;
  __shared__ PBox cbox[64];
  __shared__ float cf[64][5];   // fp32 copies for the screening pass: x1, y1, x2 + 1, y2 + 1, area
  const int t = threadIdx.x;
  {
    const int j = cb * 64 + t;
    if (j < n) {
      const PBox p = load_pbox(boxes + 4 * (int64_t)j);
      cbox[t] = p;
      cf[t][0] = (float)p.x1; cf[t][1] = (float)p.y1; cf[t][2] = (float)(p.x2 + 1); cf[t][3] = (float)(p.y2 + 1);
      cf[t][4] = (float)p.area;
    }
  }
  __syncthreads();
  const int i = rb * 64 + t;
  unsigned long long bits = 0ull;
  // Screening in fp32: with pixel coordinates below 2^13 (rounding <= 5e-4 px per corner) and sides >= 1 px (the +1
  // convention) the fp32 overlap is within ~2.5e-3 of the fp64 one for the smallest boxes and ~1e-5 for typical ones, so
  // only pairs within kMargin of the threshold (and NaNs) take the exact fp64 path of the reference. The error grows
  // with the coordinates (~1e-2 at 1.2e5 px), so `screen` is 0 for images with a side above kFrcnnScreenMaxSide (the
  // clip keeps coordinates <= side - 1): the bounds become -inf / +inf and every pair takes the fp64 path.
  // tests/test_filter_replays.py replays this screen in numpy over the whole screened domain.
  constexpr float kMargin = 4e-3f;
  const float thr_hi = screen ? (float)thr + kMargin : INFINITY, thr_lo = screen ? (float)thr - kMargin : -INFINITY;
  if (i < n) {
    const PBox my = load_pbox(boxes + 4 * (int64_t)i);
    const float mx1 = (float)my.x1, my1 = (float)my.y1, mx2 = (float)(my.x2 + 1), my2 = (float)(my.y2 + 1), ma = (float)my.area;
    for (int jj = 0; jj < 64; ++jj) {
      const int j = cb * 64 + jj;
      if (j > i && j < n) {
        const float fw = fmaxf(0.0f, fminf(mx2, cf[jj][2]) - fmaxf(mx1, cf[jj][0]));
        const float fh = fmaxf(0.0f, fminf(my2, cf[jj][3]) - fmaxf(my1, cf[jj][1]));
        const float fi = fw * fh;
        const float fo = __fdividef(fi, ma + cf[jj][4] - fi);
        if (fo > thr_hi) {
          bits |= 1ull << jj;
        } else if (!(fo < thr_lo)) {   // too close to call (or NaN): the reference's arithmetic
          const PBox o = cbox[jj];
          const double xx1 = d_max(my.x1, o.x1), yy1 = d_max(my.y1, o.y1);
          const double xx2 = d_min(my.x2, o.x2), yy2 = d_min(my.y2, o.y2);
          const double w = d_max(0.0, xx2 - xx1 + 1), h = d_max(0.0, yy2 - yy1 + 1);
          const double inter = w * h;
          const double ovr = inter / (my.area + o.area - inter);
          if (ovr >= thr) bits |= 1ull << jj;
        }
      }
    }
    if (cb != rb) mask[(int64_t)i * Ws + cb] = bits;
  }
  if (cb == rb) {
    uint32_t* dt = reinterpret_cast<uint32_t*>(diagT + (int64_t)cb * 64);   // diagonal tile: stored transposed
    const int warp = t >> 5, lane = t & 31;
    for (int jj = 0; jj < 64; ++jj) {
      const uint32_t bal = __ballot_sync(0xffffffffu, (bits >> jj) & 1ull);
      if (lane == 0) dt[jj * 2 + warp] = bal;
    }
  }
}

// fp32 path: position p of image b's visiting order holds box ix[b,p] (zeros past the valid ones); grid
// (ceil(K/256), B); npre[b] = min(num_valid[b], pre_n).
__global__ void frcnn_gather_kernel(const int32_t* __restrict__ ix, const double* __restrict__ boxes, int64_t total,
                                    int pre_n, int K, double* __restrict__ sorted, const int32_t* __restrict__ num_valid,
                                    int32_t* __restrict__ npre) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  const int b = blockIdx.y;
  const int n = min(num_valid[b], pre_n);
  if (p == 0) npre[b] = n;
  if (p >= K) return;
  const bool valid = p < n;
  const int64_t src = valid ? ix[(int64_t)b * K + p] : 0;
  OD_DBG_IDX(src, total);
  const double* bx = boxes + (int64_t)b * total * 4;
  double* o = sorted + ((int64_t)b * K + p) * 4;
#pragma unroll
  for (int c = 0; c < 4; ++c) o[c] = valid ? bx[4 * src + c] : 0.0;
}

// grid (ceil(post_n/256), B), 256 threads. Image b's kept boxes go to rows [off, off + num_kept[b]) of out
// [B*post_n,5], off = num_kept[0] + ... + num_kept[b-1], as (b,x1,y1,x2,y2); rows from the batch's total on are zero.
constexpr int kFrEmitThreads = 256;
__global__ void __launch_bounds__(kFrEmitThreads)
frcnn_emit_kernel(const double* __restrict__ sorted, const int32_t* __restrict__ keep_pos, const int32_t* __restrict__ num_kept,
                  int B, int K, int post_n, float* __restrict__ out, int32_t* __restrict__ num_out) {
  __shared__ int32_t red[2][kFrEmitThreads / 32];
  const int j = blockIdx.x * kFrEmitThreads + threadIdx.x;
  const int b = blockIdx.y;
  int before = 0, all = 0;   // < B * post_n < 2^31: the entry point caps B
  for (int q = threadIdx.x; q < B; q += kFrEmitThreads) {
    const int v = num_kept[q];
    all += v;
    before += q < b ? v : 0;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    before += __shfl_xor_sync(0xffffffffu, before, o);
    all += __shfl_xor_sync(0xffffffffu, all, o);
  }
  if ((threadIdx.x & 31) == 0) {
    red[0][threadIdx.x >> 5] = before;
    red[1][threadIdx.x >> 5] = all;
  }
  __syncthreads();
  before = 0;
  all = 0;
#pragma unroll
  for (int w = 0; w < kFrEmitThreads / 32; ++w) {
    before += red[0][w];
    all += red[1][w];
  }
  const int n = num_kept[b];
  if (j == 0) num_out[b] = n;
  if (j >= post_n) return;
  if (j < n) {
    const int p = keep_pos[(int64_t)b * post_n + j];
    OD_DBG_IDX(p, K);
    const double* s = sorted + ((int64_t)b * K + p) * 4;
    float* o = out + 5 * ((int64_t)before + j);
    o[0] = (float)b;
#pragma unroll
    for (int c = 0; c < 4; ++c) o[1 + c] = (float)s[c];
  }
  const int64_t r = (int64_t)b * post_n + j;   // every row index of the output is visited once
  if (r >= all) {
    float* o = out + 5 * r;
#pragma unroll
    for (int c = 0; c < 5; ++c) o[c] = 0.0f;
  }
}

struct FrcnnWs {
  int32_t* counters;   // [3][B]: #valid, npre, num_kept of every image (nms_scan_launch reads [B] arrays)
  Key128* keys;
  double* boxes;
  double* sorted;
  int32_t* keep_pos;
  unsigned long long* mask;
  unsigned long long* diagT;
  float* fscore;
  int32_t* ix;
  void* topk_ws;
  size_t topk_bytes;
};
static size_t carve_frcnn_ws(Workspace& w, int64_t B, int64_t total, int64_t K, int64_t post_n, FrcnnWs* out) {
  FrcnnWs f;
  const int64_t W = (K + 63) / 64;
  f.counters = w.take<int32_t>((size_t)(3 * B));
  f.keys = w.take<Key128>((size_t)(B * total));
  f.boxes = w.take<double>((size_t)(B * 4 * total));
  f.sorted = w.take<double>((size_t)(B * 4 * K));
  f.keep_pos = w.take<int32_t>((size_t)(B * post_n));
  f.mask = w.take<unsigned long long>((size_t)(B * K * nms_mask_stride(K)));
  f.diagT = w.take<unsigned long long>((size_t)(B * W * 64));
  f.fscore = w.take<float>((size_t)(B * total));
  f.ix = w.take<int32_t>((size_t)(B * K));
  f.topk_bytes = topk_workspace_bytes(B, total, K);
  f.topk_ws = w.take<char>(f.topk_bytes);
  if (out) *out = f;
  return w.off + 256;
}

}  // namespace od

using namespace od;

extern "C" {

size_t od_frcnn_proposal_workspace_bytes_batch(int64_t batch, int64_t fh, int64_t fw, const od_frcnn_params* p) {
  if (!p || batch < 0 || batch > OD_FRCNN_MAX_BATCH || fh < 0 || fw < 0) return 0;
  const int64_t total = fh * fw * p->num_anchors;
  const int64_t K = total < p->pre_nms_top_n ? total : p->pre_nms_top_n;
  Workspace w(nullptr, 0);
  return carve_frcnn_ws(w, batch, total, K, p->post_nms_top_n, nullptr);
}

size_t od_frcnn_proposal_workspace_bytes(int64_t fh, int64_t fw, const od_frcnn_params* p) {
  return od_frcnn_proposal_workspace_bytes_batch(1, fh, fw, p);
}

int od_frcnn_proposal_forward(const DLTensor* rpn_box_class_prob, const DLTensor* rpn_bbox, const od_frcnn_params* params,
                              DLTensor* proposals, DLTensor* num_out, void* ws, size_t ws_bytes, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (!params) OD_FAIL(OD_ERR_NULL, "params is NULL");
  if (!rpn_box_class_prob) OD_FAIL(OD_ERR_NULL, "rpn_box_class_prob is NULL");   // its dtype selects that of rpn_bbox
  const bool f64 = rpn_box_class_prob->dtype.bits == 64;
  const int na = params->num_anchors;
  if (na < 1 || na > 16) OD_FAIL(OD_ERR_PARAM, "num_anchors must be in [1,16]");
  if (params->image_h < 1 || params->image_w < 1) OD_FAIL(OD_ERR_PARAM, "image_h and image_w must be >= 1");
  const int64_t post_n = params->post_nms_top_n;
  if (post_n < 0 || params->pre_nms_top_n < 0) OD_FAIL(OD_ERR_PARAM, "negative top-n");
  DeviceScope scope;
  // the batch size is read from rpn_box_class_prob; every other tensor is checked against it
  OD_CHECK(check_tensor(rpn_box_class_prob, "rpn_box_class_prob", f64 ? F64 : F32, {kAny, kAny, kAny, 2 * na}, f64 ? 8 : 4, scope));
  const int64_t B = rpn_box_class_prob->shape[0], fh = rpn_box_class_prob->shape[1], fw = rpn_box_class_prob->shape[2];
  // grid y / z extents are at most 65535, and output rows are int32 indices
  if (B > OD_FRCNN_MAX_BATCH)
    OD_FAIL(OD_ERR_PARAM, "rpn_box_class_prob: batch %lld > %d images", (long long)B, OD_FRCNN_MAX_BATCH);
  if (B * post_n > INT32_MAX)
    OD_FAIL(OD_ERR_PARAM, "batch %lld x post_nms_top_n %lld proposal rows exceed 2^31 - 1", (long long)B, (long long)post_n);
  OD_CHECK(check_tensor(rpn_bbox, "rpn_bbox", f64 ? F64 : F32, {B, fh, fw, 4 * na}, f64 ? 8 : 4, scope));
  OD_CHECK(check_tensor(proposals, "proposals", F32, {B * post_n, 5}, 4, scope));
  OD_CHECK(check_tensor(num_out, "num_out", I32, {B}, 4, scope));
  const int64_t total = fh * fw * na;
  const int64_t K = total < params->pre_nms_top_n ? total : params->pre_nms_top_n;
  if (post_n == 0 || B == 0) return OD_OK;
  if (!ws) OD_FAIL(OD_ERR_WORKSPACE, "workspace is NULL");
  Workspace w(ws, ws_bytes);
  FrcnnWs f;
  carve_frcnn_ws(w, B, total, K, post_n, &f);
  if (!w.ok()) OD_FAIL(OD_ERR_WORKSPACE, "workspace %zu < %zu bytes", ws_bytes, w.off);
  int32_t* num_valid = f.counters;
  int32_t* npre = f.counters + B;
  int32_t* num_kept = f.counters + 2 * B;
  OD_CUDA(cudaMemsetAsync(f.counters, 0, (size_t)(3 * B) * sizeof(int32_t), st));
  FrcnnDev d;
  d.feat_stride = params->feat_stride; d.image_h = params->image_h; d.image_w = params->image_w;
  d.min_box_hw = params->min_box_hw; d.num_anchors = na; d.fw = (int32_t)fw;
  for (int i = 0; i < 4 * na; ++i) d.base[i] = params->base_anchors[i];
  const dim3 dgrid((unsigned)((total + 255) / 256 > 0 ? (total + 255) / 256 : 1), (unsigned)B);
  if (f64)
    frcnn_decode_kernel<double><<<dgrid, 256, 0, st>>>(dptr<double>(rpn_box_class_prob), dptr<double>(rpn_bbox), d, total, f.boxes, f.keys, num_valid, nullptr);
  else
    frcnn_decode_kernel<float><<<dgrid, 256, 0, st>>>(dptr<float>(rpn_box_class_prob), dptr<float>(rpn_bbox), d, total, f.boxes, f.keys, num_valid, f.fscore);
  OD_LAUNCH_CHECK("frcnn_decode_kernel");
  const int W = (int)((K + 63) / 64);
  if (K > 0) {
    if (f64) {   // fp64 scores: 128-bit keys, rank sort
      const dim3 grid((unsigned)((total + kFrRankMine - 1) / kFrRankMine), (unsigned)B);
      frcnn_rank_gather_kernel<<<grid, kFrRankThreads, 0, st>>>(f.keys, f.boxes, total, params->pre_nms_top_n, (int)K, f.sorted,
                                                                num_valid, npre);
      OD_LAUNCH_CHECK("frcnn_rank_gather_kernel");
    } else {     // fp32 scores: the radix-select top-k of the Mask R-CNN path, filtered-out boxes at -inf
      OD_CHECK(topk_launch(f.fscore, B, total, total, 1, K, f.ix, nullptr, f.topk_ws, f.topk_bytes, st));
      const dim3 grid((unsigned)((K + 255) / 256), (unsigned)B);
      frcnn_gather_kernel<<<grid, 256, 0, st>>>(f.ix, f.boxes, total, params->pre_nms_top_n, (int)K, f.sorted, num_valid, npre);
      OD_LAUNCH_CHECK("frcnn_gather_kernel");
    }
    const dim3 grid((unsigned)W, (unsigned)W, (unsigned)B);
    const int screen = params->image_h <= kFrcnnScreenMaxSide && params->image_w <= kFrcnnScreenMaxSide;
    frcnn_mask_kernel<<<grid, 64, 0, st>>>(f.sorted, npre, (int)K, W, (int)nms_mask_stride(K), params->nms_threshold, screen,
                                           f.mask, f.diagT);
    OD_LAUNCH_CHECK("frcnn_mask_kernel");
  }
  OD_CHECK(nms_scan_launch(f.mask, f.diagT, npre, B, K, nms_mask_stride(K), post_n, f.keep_pos, num_kept, nullptr, st));
  const dim3 egrid((unsigned)((post_n + kFrEmitThreads - 1) / kFrEmitThreads), (unsigned)B);
  frcnn_emit_kernel<<<egrid, kFrEmitThreads, 0, st>>>(f.sorted, f.keep_pos, num_kept, (int)B, (int)K, (int)post_n,
                                                      dptr<float>(proposals), dptr<int32_t>(num_out));
  OD_LAUNCH_CHECK("frcnn_emit_kernel");
  return OD_OK;
}

}  // extern "C"
