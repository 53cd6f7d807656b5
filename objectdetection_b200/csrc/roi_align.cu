// roi_align.cu — FPN level assignment + bilinear crop_and_resize gather (HBM-bound).
//
// Replaces MaskRCNN.roi_pooling (maskrcnn.py:74-187), tf.image.crop_and_resize
// (TF core/kernels/crop_and_resize_op.cc semantics) and FasterRCNN roi_pool (fastrcnn.py:22-70).
//
// Layout: feature maps NHWC fp32, so one bilinear tap is D*4 contiguous bytes (1 KiB at D=256)
// and the left/right taps of a bin are adjacent; every global access is a 16-byte vector and a
// warp reads/writes 512 contiguous bytes. The reference's per-level where/gather, concat and
// re-sort (maskrcnn.py:127-173) are not reproduced: each ROI writes straight to out[b*N+n].
//
//   crop_rows_kernel : D = 256, pool height <= 16, width <= 14 and the larger side >= 10 (the 14x14 mask-branch pooling):
//      one persistent CTA per SM, planner / issuer / consumer warps around a TMA-fed shared-memory ring of feature rows,
//      separable blend (described below).
//   roi_order_kernel : pre-pass of both kernels, the order in which the ROIs are walked (level by level, top to bottom).
//   crop_bins_kernel : every other shape. The output is one flat array of bins (roi, y, x), each D*4 contiguous bytes. A CTA owns
//      32 consecutive bins (every CTA does the same amount of work, ROI boundaries are irrelevant). Its
//      first threads build a per-bin table in shared memory: level assignment + crop_and_resize grid of the bin's
//      ROI -> image base pointer, the four tap offsets (in 16-byte units), the two lerp weights and a validity
//      flag. The main loop then is table lookup + 4 unconditional 16-byte loads per output quad (2 quads,
//      i.e. 8 loads in flight per thread), 3 lerps on packed fp32 pairs (FADD2) and one streaming
//      16-byte store. No meta kernel, no per-call allocation.
//   crop_pool_bins_kernel : FasterRCNN roi_pool = crop 14x14 fused with 2x2 max-pool, same scheme over pooled bins.
#include <cuda_bf16.h>

#include <type_traits>

#include "common.cuh"
#include "tma.cuh"

namespace od {

struct __align__(16) RoiMeta {
  const void* base;   // image (level, batch) base, an fp32 or bf16 array
  int32_t H, W;
  float in_y0, hs, in_x0, ws;  // in_y = in_y0 + y * hs   (TF: y1*(H-1) + y*height_scale)
};

struct LevelTable {
  const void* ptr[OD_MAX_LEVELS];               // NHWC maps of one dtype: fp32 or bf16
  int32_t H[OD_MAX_LEVELS];
  int32_t W[OD_MAX_LEVELS];
};

// maskrcnn.py:104-122
__device__ __forceinline__ int32_t roi_level_of(float4 r, int32_t image_h, int32_t image_w, int32_t min_level,
                                                int32_t max_level) {
  const float h = r.z - r.x;
  const float w = r.w - r.y;
  const float image_area = (float)(image_h * image_w);
  const float denom = 224.0f / sqrtf(image_area);
  const float v = sqrtf(h * w) / denom;
  const float lv = f_log(v) / f_log(2.0f);
  const float rr = rintf(lv);  // half to even
  int32_t level = (int32_t)(4u + (uint32_t)f_to_i32_x86(rr));
  level = max(level, min_level);
  level = min(level, max_level);
  return level;
}

__device__ __forceinline__ void fill_grid(RoiMeta& m, float4 box, int32_t ph, int32_t pw) {
  const float y1 = box.x, x1 = box.y, y2 = box.z, x2 = box.w;
  const float Hm1 = (float)(m.H - 1), Wm1 = (float)(m.W - 1);
  if (ph > 1) {
    m.hs = (y2 - y1) * Hm1 / (float)(ph - 1);
    m.in_y0 = y1 * Hm1;
  } else {
    m.hs = 0.0f;
    m.in_y0 = (float)(0.5 * (double)(y1 + y2) * (double)(m.H - 1));
  }
  if (pw > 1) {
    m.ws = (x2 - x1) * Wm1 / (float)(pw - 1);
    m.in_x0 = x1 * Wm1;
  } else {
    m.ws = 0.0f;
    m.in_x0 = (float)(0.5 * (double)(x1 + x2) * (double)(m.W - 1));
  }
}

__device__ __forceinline__ float4 max4(float4 a, float4 b) {
  return make_float4(f_max(a.x, b.x), f_max(a.y, b.y), f_max(a.z, b.z), f_max(a.w, b.w));
}

// ----------------------------------------------------------------------------- crop_bins_kernel
// Where a ROI comes from: mode 0 = PyramidROIAlign (level from the box, batch = roi / rois_per_image),
// mode 1 = tf.image.crop_and_resize (explicit box_ind, one image tensor in lt slot 0),
// mode 2 = FasterRCNN roi_pool: rows (batch, x1, y1, x2, y2) in pixels, divided by (image_h, image_w)
//          (fastrcnn.py:55-64), one image tensor in lt slot 0.
struct RoiSource {
  int32_t mode;
  int32_t rois_per_image;
  int32_t image_h, image_w, min_level, num_levels;
  int32_t batch;
  LevelTable lt;
  const float4* boxes;
  const int32_t* box_ind;
  const float* boxes5;
  float fimage_h, fimage_w;
  const int32_t* order;   // optional (mode 0): processing order of the ROIs, order[j] = ROI handled j-th (roi_order_kernel)
};

struct __align__(16) BinTaps {  // tap offsets from the image base, in 16-byte units
  uint32_t tl, tr, bl, br;
};
struct __align__(16) BinInfo {  // base pointer (16-byte aligned) | flag in the low bits
  uintptr_t base_flag;
  float xl, yl;
};
constexpr uintptr_t kBinSample = 0, kBinExtrapolate = 1, kBinSkip = 2;
// CTA shape of the flat-bin kernels: 32 bins per 128-thread CTA, 2 quads in flight per thread, the best of the sweeps in
// profiles/r1_crop_variants.md.
constexpr int kBinThreads = 128;
constexpr int kBinBins = 32;
constexpr int kBinUnroll = 2;

// packed fp32 pairs (sm_100 FADD2): IEEE add/sub on both halves, so results equal two scalar ops
__device__ __forceinline__ void add2(float& d0, float& d1, float a0, float a1, float b0, float b1) {
  unsigned long long ra, rb, rd;
  asm("mov.b64 %0, {%1,%2};" : "=l"(ra) : "f"(a0), "f"(a1));
  asm("mov.b64 %0, {%1,%2};" : "=l"(rb) : "f"(b0), "f"(b1));
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
  asm("mov.b64 {%0,%1}, %2;" : "=f"(d0), "=f"(d1) : "l"(rd));
}
__device__ __forceinline__ void sub2(float& d0, float& d1, float a0, float a1, float b0, float b1) {
  unsigned long long ra, rb, rd;
  asm("mov.b64 %0, {%1,%2};" : "=l"(ra) : "f"(a0), "f"(a1));
  asm("mov.b64 %0, {%1,%2};" : "=l"(rb) : "f"(b0), "f"(b1));
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
  asm("mov.b64 {%0,%1}, %2;" : "=f"(d0), "=f"(d1) : "l"(rd));
}
__device__ __forceinline__ float4 sub4p(float4 b, float4 a) {
  float4 d;
  sub2(d.x, d.y, b.x, b.y, a.x, a.y);
  sub2(d.z, d.w, b.z, b.w, a.z, a.w);
  return d;
}
// a + d * t per component, d = b - a computed by the caller. The multiply stays scalar: ptxas contracts a packed
// mul.rn.f32x2 + add.rn.f32x2 pair into FFMA2 even with -fmad=false (checked in SASS), which would change the rounding.
__device__ __forceinline__ float4 axpy4p(float4 a, float4 d, float t) {
  float4 m, r;
  m.x = __fmul_rn(d.x, t);
  m.y = __fmul_rn(d.y, t);
  m.z = __fmul_rn(d.z, t);
  m.w = __fmul_rn(d.w, t);
  add2(r.x, r.y, a.x, a.y, m.x, m.y);
  add2(r.z, r.w, a.z, a.w, m.z, m.w);
  return r;
}
// a + (b - a) * t per component, every operation individually rounded (the multiply stays scalar: ptxas would
// contract mul.f32x2 + add.f32x2 into FFMA2)
__device__ __forceinline__ float4 lerp4p(float4 a, float4 b, float t) {
  float4 d, r;
  sub2(d.x, d.y, b.x, b.y, a.x, a.y);
  sub2(d.z, d.w, b.z, b.w, a.z, a.w);
  d.x = __fmul_rn(d.x, t);
  d.y = __fmul_rn(d.y, t);
  d.z = __fmul_rn(d.z, t);
  d.w = __fmul_rn(d.w, t);
  add2(r.x, r.y, a.x, a.y, d.x, d.y);
  add2(r.z, r.w, a.z, a.w, d.z, d.w);
  return r;
}

// ----------------------------------------------------------------------------- fp32 and bf16 units
// The kernels move a feature pixel in 16-byte units: 4 fp32 channels, or 8 bf16 channels. A bf16 unit is widened to fp32
// exactly (a bf16 is the upper half of an fp32) and blended like two fp32 units, so the fp32 result does not depend on
// the map dtype. The result is stored as fp32, or rounded to the nearest bf16, ties to even (cvt.rn.bf16x2.f32).
struct float8 {                                    // the 8 channels of one bf16 unit, widened
  float4 lo, hi;
};
struct __align__(8) bf16x4 {                       // pooled output unit, fp32 maps -> bf16
  __nv_bfloat162 v[2];
};
struct __align__(16) bf16x8 {                      // pooled output unit, bf16 maps -> bf16
  __nv_bfloat162 v[4];
};
template <typename TMap> struct MapUnit;           // Raw: as loaded; Val: widened to fp32; kCh channels
template <> struct MapUnit<float> {
  using Raw = float4;
  using Val = float4;
  static constexpr int kCh = 4;
};
template <> struct MapUnit<__nv_bfloat16> {
  using Raw = uint4;
  using Val = float8;
  static constexpr int kCh = 8;
};
template <typename TMap, typename TOut> struct OutUnit;   // one map unit's channels in the pooled dtype
template <> struct OutUnit<float, float> { using T = float4; };
template <> struct OutUnit<__nv_bfloat16, float> { using T = float8; };
template <> struct OutUnit<float, __nv_bfloat16> { using T = bf16x4; };
template <> struct OutUnit<__nv_bfloat16, __nv_bfloat16> { using T = bf16x8; };

__device__ __forceinline__ float4 widen_unit(float4 v) { return v; }
__device__ __forceinline__ float8 widen_unit(uint4 v) {
  float8 r;
  r.lo = make_float4(__uint_as_float(v.x << 16), __uint_as_float(v.x & 0xFFFF0000u), __uint_as_float(v.y << 16),
                     __uint_as_float(v.y & 0xFFFF0000u));
  r.hi = make_float4(__uint_as_float(v.z << 16), __uint_as_float(v.z & 0xFFFF0000u), __uint_as_float(v.w << 16),
                     __uint_as_float(v.w & 0xFFFF0000u));
  return r;
}
__device__ __forceinline__ float4 ldg_unit(const float4* p) { return ldg_f4(p); }
__device__ __forceinline__ float8 ldg_unit(const uint4* p) { return widen_unit(__ldg(p)); }
template <typename V> __device__ __forceinline__ V splat_unit(float v);
template <> __device__ __forceinline__ float4 splat_unit<float4>(float v) { return make_float4(v, v, v, v); }
template <> __device__ __forceinline__ float8 splat_unit<float8>(float v) {
  return {make_float4(v, v, v, v), make_float4(v, v, v, v)};
}
// the fp32 blends of a bf16 unit: the same operations on both halves
__device__ __forceinline__ float8 sub4p(float8 b, float8 a) { return {sub4p(b.lo, a.lo), sub4p(b.hi, a.hi)}; }
__device__ __forceinline__ float8 axpy4p(float8 a, float8 d, float t) { return {axpy4p(a.lo, d.lo, t), axpy4p(a.hi, d.hi, t)}; }
__device__ __forceinline__ float8 lerp4p(float8 a, float8 b, float t) { return {lerp4p(a.lo, b.lo, t), lerp4p(a.hi, b.hi, t)}; }
// streaming stores of one output unit
__device__ __forceinline__ uint32_t bf16x2_rn(float lo, float hi) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ void st_unit(float4* p, float4 v) { stg_cs_f4(p, v); }
__device__ __forceinline__ void st_unit(float8* p, float8 v) {
  stg_cs_f4(&p->lo, v.lo);
  stg_cs_f4(&p->hi, v.hi);
}
__device__ __forceinline__ void st_unit(bf16x4* p, float4 v) {
  __stcs(reinterpret_cast<uint2*>(p), make_uint2(bf16x2_rn(v.x, v.y), bf16x2_rn(v.z, v.w)));
}
__device__ __forceinline__ void st_unit(bf16x8* p, float8 v) {
  __stcs(reinterpret_cast<uint4*>(p), make_uint4(bf16x2_rn(v.lo.x, v.lo.y), bf16x2_rn(v.lo.z, v.lo.w),
                                                 bf16x2_rn(v.hi.x, v.hi.y), bf16x2_rn(v.hi.z, v.hi.w)));
}

// One entry of a CTA's bin table: level assignment + crop_and_resize grid of ROI `roi`, sampled at bin (y, x) ->
// base pointer | flag, the four tap offsets (16-byte units, D4 of them per pixel) and the two lerp weights.
template <typename TMap>
__device__ __forceinline__ void bin_table_entry(const RoiSource& src, int64_t roi, int32_t y, int32_t x, bool first_bin,
                                                int32_t ph, int32_t pw, int32_t D4, int32_t* __restrict__ level_out,
                                                BinTaps* tp_out, BinInfo* bi_out) {
  constexpr int64_t kUnitElems = 16 / sizeof(TMap);
  float4 box;
  RoiMeta m;
  uintptr_t flag = kBinSample;
  if (src.mode == 0) {
    box = __ldg(&src.boxes[roi]);
    const int32_t level = roi_level_of(box, src.image_h, src.image_w, src.min_level, src.min_level + src.num_levels - 1);
    const int32_t l = level - src.min_level;
    m.H = src.lt.H[l];
    m.W = src.lt.W[l];
    m.base = static_cast<const TMap*>(src.lt.ptr[l]) + (roi / src.rois_per_image) * ((int64_t)m.H * m.W * D4 * kUnitElems);
    if (level_out && first_bin) level_out[roi] = level;
  } else {
    int32_t b;
    if (src.mode == 1) {
      box = __ldg(&src.boxes[roi]);
      b = __ldg(&src.box_ind[roi]);
    } else {
      const float* p = src.boxes5 + 5 * roi;
      b = (int32_t)p[0];
      box = make_float4(p[2] / src.fimage_h, p[1] / src.fimage_w, p[4] / src.fimage_h, p[3] / src.fimage_w);
    }
    m.H = src.lt.H[0];
    m.W = src.lt.W[0];
    if (b >= 0 && b < src.batch) {
      m.base = static_cast<const TMap*>(src.lt.ptr[0]) + (int64_t)b * ((int64_t)m.H * m.W * D4 * kUnitElems);
    } else {  // box_ind out of range: TF skips the crop, the output rows are left untouched
      m.base = src.lt.ptr[0];
      flag = kBinSkip;
    }
  }
  fill_grid(m, box, ph, pw);
  const float in_y = m.in_y0 + (float)y * m.hs;
  const float in_x = m.in_x0 + (float)x * m.ws;
  const bool ok = (in_y >= 0.0f) && (in_y <= (float)(m.H - 1)) && (in_x >= 0.0f) && (in_x <= (float)(m.W - 1));
  BinTaps tp = {0u, 0u, 0u, 0u};
  BinInfo bi;
  bi.xl = 0.0f;
  bi.yl = 0.0f;
  if (ok) {
    const float fy = floorf(in_y), fx = floorf(in_x);
    const uint32_t top = (uint32_t)fy, bot = (uint32_t)ceilf(in_y);
    const uint32_t left = (uint32_t)fx, right = (uint32_t)ceilf(in_x);
    const uint32_t W = (uint32_t)m.W, d4 = (uint32_t)D4;
    OD_DBG_ASSERT(bot < (uint32_t)m.H && right < W && top <= bot && left <= right, "bilinear tap outside the feature map");
    tp.tl = (top * W + left) * d4;
    tp.tr = (top * W + right) * d4;
    tp.bl = (bot * W + left) * d4;
    tp.br = (bot * W + right) * d4;
    bi.xl = in_x - fx;
    bi.yl = in_y - fy;
  } else if (flag == kBinSample) {
    flag = kBinExtrapolate;
  }
  bi.base_flag = reinterpret_cast<uintptr_t>(m.base) | flag;
  *tp_out = tp;
  *bi_out = bi;
}

// D4: 16-byte units per pixel (D / 4 fp32 or D / 8 bf16 channels); `out` is addressed in the same units
template <typename TMap, typename TOut, int BINS, int UNROLL, bool POW2, bool ORDERED>
__device__ __forceinline__ void crop_bins_body(const RoiSource& src, int64_t total_bins, int32_t bins_per_roi, int32_t ph,
                                               int32_t pw, int32_t D4, int32_t lgD4, float extrap,
                                               typename OutUnit<TMap, TOut>::T* __restrict__ out,
                                               int32_t* __restrict__ level_out) {
  using Raw = typename MapUnit<TMap>::Raw;
  using Val = typename MapUnit<TMap>::Val;
  using Out = typename OutUnit<TMap, TOut>::T;
  pdl_prologue();
  __shared__ BinTaps s_taps[BINS];
  __shared__ BinInfo s_info[BINS];
  __shared__ uint32_t s_obin[ORDERED ? BINS : 1];    // ORDERED: output bin of table entry i (ROIs are walked in src.order)
  const int32_t t = threadIdx.x;
  const int64_t bin0 = (int64_t)blockIdx.x * BINS;
  const int32_t nb = (int32_t)min((int64_t)BINS, total_bins - bin0);

  for (int32_t i = t; i < nb; i += kBinThreads) {
    const int64_t fb = bin0 + i;
    int64_t roi = fb / bins_per_roi;
    const int32_t bin = (int32_t)(fb - roi * bins_per_roi);
    bool valid = true;
    if (ORDERED) {
      roi = __ldg(&src.order[roi]);
      valid = roi >= 0 && roi * bins_per_roi < total_bins;     // a caller-supplied order is not trusted: bad entry = no output
      if (!valid) roi = 0;
      s_obin[i] = (uint32_t)(roi * bins_per_roi + bin);
    }
    const int32_t y = bin / pw;
    bin_table_entry<TMap>(src, roi, y, bin - y * pw, bin == 0 && valid, ph, pw, D4, valid ? level_out : nullptr, &s_taps[i],
                          &s_info[i]);
    if (ORDERED && !valid) s_info[i].base_flag = (s_info[i].base_flag & ~(uintptr_t)3) | kBinSkip;
  }
  __syncthreads();

  const int32_t total = nb * D4;
  Out* __restrict__ o = out + bin0 * D4;
  const Val ext4 = splat_unit<Val>(extrap);
  for (int32_t e0 = t; e0 < total; e0 += kBinThreads * UNROLL) {
    Raw tl[UNROLL], tr[UNROLL], bl[UNROLL], br[UNROLL];   // bf16 units are widened at the blend: half the registers
    float xl[UNROLL], yl[UNROLL];
    uint32_t fl[UNROLL];
    Out* op[UNROLL];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      const int32_t e = min(e0 + u * kBinThreads, total - 1);  // clamped: loads are unconditional
      const int32_t bin = POW2 ? (e >> lgD4) : (e / D4);
      const uint32_t c = (uint32_t)(POW2 ? (e & (D4 - 1)) : (e - bin * D4));
      OD_DBG_IDX(bin, BINS);
      const BinTaps tp = s_taps[bin];
      const BinInfo bi = s_info[bin];
      const Raw* __restrict__ base = reinterpret_cast<const Raw*>(bi.base_flag & ~(uintptr_t)15);
      fl[u] = (uint32_t)(bi.base_flag & 3u);
      xl[u] = bi.xl;
      yl[u] = bi.yl;
      op[u] = ORDERED ? out + ((int64_t)s_obin[bin] * D4 + c) : o + e;
      tl[u] = __ldg(base + (tp.tl + c));
      tr[u] = __ldg(base + (tp.tr + c));
      bl[u] = __ldg(base + (tp.bl + c));
      br[u] = __ldg(base + (tp.br + c));
    }
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      const int32_t e = e0 + u * kBinThreads;
      const Val top = lerp4p(widen_unit(tl[u]), widen_unit(tr[u]), xl[u]);
      const Val bot = lerp4p(widen_unit(bl[u]), widen_unit(br[u]), xl[u]);
      Val v = lerp4p(top, bot, yl[u]);
      if (fl[u] == (uint32_t)kBinExtrapolate) v = ext4;
      if (e < total && fl[u] != (uint32_t)kBinSkip) st_unit(op[u], v);
    }
  }
}

template <int BINS, int UNROLL, bool POW2, bool ORDERED>
__global__ void __launch_bounds__(kBinThreads, 1)
crop_bins_kernel(RoiSource src, int64_t total_bins, int32_t bins_per_roi, int32_t ph, int32_t pw, int32_t D4,
                 int32_t lgD4, float extrap, float4* __restrict__ out, int32_t* __restrict__ level_out) {
  crop_bins_body<float, float, BINS, UNROLL, POW2, ORDERED>(src, total_bins, bins_per_roi, ph, pw, D4, lgD4, extrap, out,
                                                            level_out);
}
// bf16 maps and / or a bf16 output: the same body, an overload of the same name (the fp32 kernel above keeps its name)
template <typename TMap, typename TOut, int BINS, int UNROLL, bool POW2, bool ORDERED>
__global__ void __launch_bounds__(kBinThreads, 1)
crop_bins_kernel(RoiSource src, int64_t total_bins, int32_t bins_per_roi, int32_t ph, int32_t pw, int32_t D4,
                 int32_t lgD4, float extrap, typename OutUnit<TMap, TOut>::T* __restrict__ out,
                 int32_t* __restrict__ level_out) {
  crop_bins_body<TMap, TOut, BINS, UNROLL, POW2, ORDERED>(src, total_bins, bins_per_roi, ph, pw, D4, lgD4, extrap, out,
                                                          level_out);
}

// ----------------------------------------------------------------------------- roi_order_kernel
// Proposals arrive sorted by score, i.e. in random spatial order, while overlapping ROIs read the same feature pixels:
// walked in index order the ROIs of one image pull ~1.4x the pyramid through DRAM (L2 holds the write stream too),
// walked level by level and top to bottom every pixel is fetched once (profiles/r2_roialign.md). One CTA per image
// buckets its ROIs by (pyramid level, 32 bands of the box centre's y) with a shared-memory counting sort and writes the
// processing order; the order inside a bucket is whatever the atomics produce (any order gives the same output).
constexpr int kOrderBands = 32;
constexpr int kOrderThreads = 1024;
constexpr int kOrderPerThread = 4;               // up to 4096 ROIs per image; beyond that the order is not used
__global__ void __launch_bounds__(kOrderThreads)
roi_order_kernel(const float4* __restrict__ boxes, int32_t N, int32_t image_h, int32_t image_w, int32_t min_level,
                 int32_t num_levels, int32_t* __restrict__ order) {
  pdl_prologue();
  __shared__ int32_t s_cnt[OD_MAX_LEVELS * kOrderBands];
  __shared__ int32_t s_base[OD_MAX_LEVELS * kOrderBands];
  const int32_t t = threadIdx.x, b = blockIdx.x;
  const int32_t nb = num_levels * kOrderBands;
  for (int32_t i = t; i < nb; i += kOrderThreads) s_cnt[i] = 0;
  __syncthreads();
  int32_t key[kOrderPerThread], pos[kOrderPerThread];
#pragma unroll
  for (int j = 0; j < kOrderPerThread; ++j) {
    const int32_t n = t + j * kOrderThreads;
    key[j] = -1;
    if (n < N) {
      const float4 bx = __ldg(&boxes[(int64_t)b * N + n]);
      // the order only steers locality (any order gives the same output), so the level key may be approximate: fast
      // fp32 log2 (MUFU) instead of the correctly rounded fp64 log of roi_level_of, 1.5 us less on the serial path
      const float v = sqrtf((bx.z - bx.x) * (bx.w - bx.y)) * sqrtf((float)(image_h * image_w)) * (1.0f / 224.0f);
      const float lf = 4.0f + rintf(__log2f(v));                                     // NaN / <= 0 -> NaN or -inf
      int32_t lv = (lf >= (float)min_level) ? (lf < (float)(min_level + num_levels) ? (int32_t)lf : min_level + num_levels - 1)
                                           : min_level;                             // NaN -> min_level
      lv -= min_level;
      const float yc = 0.5f * (bx.x + bx.z) * (float)kOrderBands;
      const int32_t band = (yc >= 0.0f) ? (yc < (float)kOrderBands ? (int32_t)yc : kOrderBands - 1) : 0;   // NaN -> 0
      key[j] = lv * kOrderBands + band;
      OD_DBG_IDX(key[j], nb);
      pos[j] = atomicAdd(&s_cnt[key[j]], 1);
    }
  }
  __syncthreads();
  if (t < 32) {                                   // exclusive scan of <= 256 bucket counts, 8 per lane
    int32_t c[OD_MAX_LEVELS * kOrderBands / 32], sum = 0;
#pragma unroll
    for (int i = 0; i < OD_MAX_LEVELS * kOrderBands / 32; ++i) {
      const int32_t k = t * (OD_MAX_LEVELS * kOrderBands / 32) + i;
      c[i] = k < nb ? s_cnt[k] : 0;
      sum += c[i];
    }
    int32_t incl = sum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int32_t v = __shfl_up_sync(0xffffffffu, incl, d);
      if (t >= d) incl += v;
    }
    int32_t run = incl - sum;
#pragma unroll
    for (int i = 0; i < OD_MAX_LEVELS * kOrderBands / 32; ++i) {
      const int32_t k = t * (OD_MAX_LEVELS * kOrderBands / 32) + i;
      if (k < nb) s_base[k] = run;
      run += c[i];
    }
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < kOrderPerThread; ++j)
    if (key[j] >= 0) {
      OD_DBG_IDX(s_base[key[j]] + pos[j], N);
      order[(int64_t)b * N + s_base[key[j]] + pos[j]] = b * N + t + j * kOrderThreads;
    }
}

// ----------------------------------------------------------------------------- crop_rows_kernel
// The TMA-staged, separable form of the same gather (D = 256, pool height <= 16, pool width <= 14). ONE persistent CTA per
// SM (512 threads, ~100 registers free to use, a 176 KiB ring), drawing ROIs from a ticket counter (in the order
// roi_order_kernel wrote), with three kinds of warps that only meet through mbarriers:
//
//   planner   (1 warp) turns ROI geometry into a PLAN, up to kRowsPlans ROIs ahead of the consumers. crop_and_resize samples
//             a ROI on a separable grid - bin (y, x) blends feature rows top(y)/bot(y) and columns left(x)/right(x). With a
//             non-negative step the taps are monotone, so the DISTINCT rows the ROI needs, in first-use = ascending order,
//             are ranked 0..nr-1 with two ballots and a popcount (lanes 0-15: y samples, lanes 16-31: x samples); the
//             columns likewise, consecutive column ranks merged into runs of adjacent pixels. A 14x14 crop of an 8-pixel
//             ROI needs 9 rows of 9 pixels instead of 784 taps. The ticket is drawn two plans ahead and the box fetched one
//             plan ahead, so no global round trip sits between two plans.
//   issuer    (1 warp) streams the ranked rows of ROI after ROI into one shared-memory BYTE ring: one cp.async.bulk per
//             (row, column run) - NHWC makes a run of pixels one contiguous block of len KiB - completion counted in bytes
//             on the entry's `full` mbarrier; space is reclaimed in FIFO order as all consumer warps arrive on an entry's
//             `empty` mbarrier. The ring never drains between ROIs; bytes in flight are set by the ring size, not by
//             registers or occupancy - the deeper the ring, the faster the kernel (profiles/r2_roialign.md).
//   consumers (one warp per x bin, lane = channel quads `lane` and `lane + 32`) walk the ROW RANKS: the output rows whose
//             top row has rank k are contiguous (yfirst), their bottom row is rank k or k+1. On first use a row is blended
//             left/right straight from the ring (4 LDS.128) into registers and the entry released; every output row is then
//             one lerp between the two cached rows and two streaming 16-byte stores. Every feature pixel is read once from
//             L2 per ROI and each x-blend is computed once per (row, x) instead of once per bin.
//   ROIs the plan cannot serve (flipped / NaN / partly outside boxes) take a per-bin path with direct loads on the
//   consumer warps.
// Arithmetic per output value is the reference's (crop_and_resize_op.cc): top = tl + (tr - tl) * xl, bot likewise,
// out = top + (bot - top) * yl, so the results are bit-identical to crop_bins_kernel and to the oracle.
// Measured and slower (profiles/r2_roialign.md): output rows written by bulk shared->global copies (2-8 %), one channel
// quad per lane with two warps per x bin, two 64-register CTAs per SM with half the ring each (10 %), L2 evict_last
// hints on the ring copies and an L2 prefetch of the planned rows.
constexpr int kRowsThreads = 512;
constexpr int kRowsMaxPool = 16;                // plan tables: pool height <= 16 (the width is capped by kRowsMaxWidth)
constexpr int kRowsMaxWidth = kRowsThreads / 32 - 2;   // one consumer warp per x bin next to the issuer and the planner
constexpr int kRowsMinPool = 10;                // smaller pools leave too few consumer warps per SM: 7x7 takes 0.063 ms
                                                // here against 0.043 ms in crop_bins_kernel (profiles/r2_roialign.md)
constexpr int kRowsEntries = 32;                // outstanding ring entries (one feature row each)
constexpr int kRowsPlans = 3;                   // plans in flight
constexpr int kRowsD4 = 64;                     // D = 256 floats = 64 quads = 1 KiB per pixel
constexpr uint32_t kRowsPixelBytes = 1024;      // fp32 maps; a bf16 pixel is 512 bytes (32 units of 8 channels)
template <typename TMap> constexpr int kRowsUnits = 4 * kRowsD4 / MapUnit<TMap>::kCh;   // 16-byte units per pixel
// Ring size: 176 KiB. The kernel alone is ~1 % faster with everything an SM has (221 KiB), but leaving ~45 KiB lets the
// small CTAs of concurrently running kernels (the other steps' proposal front and 7x7 ROIAlign) become resident next to
// it, which is worth 8 % of whole-step throughput (profiles/r2_roialign.md).
constexpr uint32_t kRowsRingBytes = 176 * 1024;
// A row may have to skip the tail of the ring (it never straddles the end): row + skipped tail must fit an EMPTY ring,
// which holds for every head position only if a row is at most half the ring. A row holds the distinct columns of one
// ROI, at most two per x sample. (The fp32 pixel is the larger one.)
static_assert(2u * (2 * kRowsMaxWidth) * kRowsPixelBytes <= kRowsRingBytes, "a ring row can exceed half the ring");

struct RowsPlan {
  int2 ytab[kRowsMaxPool + 2];                  // ring mode, per y: {y_lerp bits, top row == bottom row}; two pad entries
  int32_t yfirst[2 * kRowsMaxPool + 1];         // ring mode: first y whose TOP row has rank >= k (y's of rank k are contiguous)
  int32_t y_top[kRowsMaxPool], y_bot[kRowsMaxPool], y_ok[kRowsMaxPool];
  float y_lerp[kRowsMaxPool];
  int32_t x_left[kRowsMaxPool], x_right[kRowsMaxPool], x_cl[kRowsMaxPool], x_cr[kRowsMaxPool], x_ok[kRowsMaxPool];
  float x_lerp[kRowsMaxPool];
  int32_t rows[2 * kRowsMaxPool];               // feature row of row-rank k
  int32_t run_col[kRowsMaxPool], run_rank[kRowsMaxPool], run_len[kRowsMaxPool];
  int32_t nr, ncols, nruns, mode;
  int32_t W;
  uint32_t row_bytes;                           // ncols pixels: one ring entry
  int64_t roi;
  const void* base;
};
// ring: every bin of the ROI has four valid taps and the grid steps are non-negative (the streaming fast path);
// flat: anything else (extrapolated bins, flipped / NaN boxes) - per-bin direct loads;
// skip: box_ind out of range, the crop is left untouched; done: no ROI left for this CTA.
constexpr int kRowsRing = 0, kRowsFlat = 1, kRowsSkip = 2, kRowsDone = 3;

struct RowsShared {
  RowsPlan plan[kRowsPlans];
  int32_t cols[2 * kRowsMaxPool];               // planner scratch
  uint32_t entry_fp[kRowsEntries];              // ring bytes an entry occupies incl. wrap padding (issuer only)
  unsigned long long full[kRowsEntries], empty[kRowsEntries], plan_full[kRowsPlans], plan_empty[kRowsPlans];
};

// geometry of one ROI (level assignment, image base, sampling grid) from its preloaded box (and batch index in
// crop_and_resize mode); returns the kBin* flag
template <typename TMap>
__device__ __forceinline__ uintptr_t roi_geometry(const RoiSource& src, int64_t roi, float4 box, int32_t b, int32_t ph,
                                                  int32_t pw, RoiMeta& m, int32_t* level) {
  uintptr_t flag = kBinSample;
  constexpr int64_t D = 4 * kRowsD4;
  if (src.mode == 0) {
    *level = roi_level_of(box, src.image_h, src.image_w, src.min_level, src.min_level + src.num_levels - 1);
    const int32_t l = *level - src.min_level;
    m.H = src.lt.H[l];
    m.W = src.lt.W[l];
    m.base = static_cast<const TMap*>(src.lt.ptr[l]) + (int64_t)((uint32_t)roi / (uint32_t)src.rois_per_image) * ((int64_t)m.H * m.W * D);
  } else {
    m.H = src.lt.H[0];
    m.W = src.lt.W[0];
    const TMap* base = static_cast<const TMap*>(src.lt.ptr[0]);
    if (b >= 0 && b < src.batch) base += (int64_t)b * ((int64_t)m.H * m.W * D);
    else flag = kBinSkip;
    m.base = base;
  }
  fill_grid(m, box, ph, pw);
  return flag;
}

// One warp builds the plan of one ROI, all lanes busy: lanes 0-15 own the y samples, lanes 16-31 the x samples.
// With a non-negative grid step the tap sequence lo(0) <= hi(0), lo(1) <= hi(1), ... is non-decreasing and
// hi - lo is 0 or 1, so a tap is NEW (not seen before) exactly when it differs from both taps of the previous
// sample; first-use order is ascending order, the rank of a new tap is the number of new taps before it (two
// ballots and a popcount) and a repeated tap is the largest or second largest value seen so far.
template <typename TMap>
__device__ __forceinline__ void rows_make_plan(const RoiSource& src, int64_t roi, float4 box, int32_t bidx, int32_t ph,
                                               int32_t pw, int32_t lane, RowsPlan& P, RowsShared& S, int32_t* level_out) {
  RoiMeta m;
  int32_t level = 0;
  const uintptr_t flag = roi_geometry<TMap>(src, roi, box, bidx, ph, pw, m, &level);
  const bool mono = (m.hs >= 0.0f) && (m.ws >= 0.0f);
  const int32_t half = lane >> 4, i = lane & 15;
  const int32_t n = half ? pw : ph;
  const bool valid = i < n;
  const float in = half ? (m.in_x0 + (float)i * m.ws) : (m.in_y0 + (float)i * m.hs);
  const float lim = (float)((half ? m.W : m.H) - 1);
  const bool ok = !valid || ((in >= 0.0f) && (in <= lim));
  const float fl = floorf(in);
  const int32_t lo = (valid && ok) ? (int32_t)fl : 0;
  const int32_t hi = (valid && ok) ? (int32_t)ceilf(in) : 0;
  const float lerp = (valid && ok) ? in - fl : 0.0f;
  if (valid) {                                      // the per-bin tables (the flat path reads them)
    if (half) {
      P.x_ok[i] = ok;
      P.x_left[i] = lo;
      P.x_right[i] = hi;
      P.x_lerp[i] = lerp;
    } else {
      P.y_ok[i] = ok;
      P.y_top[i] = lo;
      P.y_bot[i] = hi;
      P.y_lerp[i] = lerp;
    }
  }
  const bool all_ok = __all_sync(0xffffffffu, ok);  // every bin has four valid taps
  const int32_t mode = (flag == kBinSkip) ? kRowsSkip : ((all_ok && mono) ? kRowsRing : kRowsFlat);
  if (mode == kRowsRing) {
    const int32_t plo = __shfl_up_sync(0xffffffffu, lo, 1), phi = __shfl_up_sync(0xffffffffu, hi, 1);
    const bool new_lo = valid && (i == 0 || (lo != plo && lo != phi));
    const bool new_hi = valid && hi != lo && (i == 0 || hi != phi);
    const uint32_t hm = half ? 0xFFFF0000u : 0x0000FFFFu;
    const uint32_t ml = __ballot_sync(0xffffffffu, new_lo) & hm, mh = __ballot_sync(0xffffffffu, new_hi) & hm;
    const uint32_t below = hm & ((1u << lane) - 1u);
    const int32_t c = __popc(ml & below) + __popc(mh & below);      // distinct taps before this sample
    const int32_t r_lo = new_lo ? c : (lo == phi ? c - 1 : c - 2);
    const int32_t c2 = c + (new_lo ? 1 : 0);
    const int32_t r_hi = (hi == lo) ? r_lo : (new_hi ? c2 : c2 - 1);
    const int32_t cnt = __popc(ml) + __popc(mh);                    // distinct taps of this half
    int32_t* vals = half ? S.cols : P.rows;
    OD_DBG_ASSERT(!valid || (r_lo >= 0 && r_lo <= r_hi && r_hi < cnt && cnt <= 2 * kRowsMaxPool), "tap rank outside the plan");
    if (new_lo) vals[r_lo] = lo;
    if (new_hi) vals[r_hi] = hi;
    if (valid) {
      if (half) {
        P.x_cl[i] = r_lo;
        P.x_cr[i] = r_hi;
      } else {
        P.ytab[i] = make_int2(__float_as_int(lerp), r_hi == r_lo ? 1 : 0);
      }
    }
    {   // lane k: how many y's blend a top row of rank < k (ranks are <= 31, entry 32 is the pool height)
      int32_t before = 0;
      for (int32_t y = 0; y < ph; ++y) before += (__shfl_sync(0xffffffffu, r_lo, y) < lane) ? 1 : 0;
      P.yfirst[lane] = before;
      if (lane == 0) P.yfirst[32] = ph;
    }
    const int32_t nc = __shfl_sync(0xffffffffu, cnt, 16), nr = __shfl_sync(0xffffffffu, cnt, 0);
    __syncwarp();
    // distinct columns -> runs of adjacent pixels (one bulk copy each): lane k looks at column rank k
    const int32_t ck = lane < nc ? S.cols[lane] : 0;
    const int32_t cp = __shfl_up_sync(0xffffffffu, ck, 1);
    const bool start = lane < nc && (lane == 0 || ck != cp + 1);
    const uint32_t sm = __ballot_sync(0xffffffffu, start);
    if (start) {
      const uint32_t le = (2u << lane) - 1u;        // lanes <= this one (wraps to all ones for lane 31)
      const int32_t j = __popc(sm & le) - 1;
      OD_DBG_IDX(j, kRowsMaxPool);
      const uint32_t rest = sm & ~le;
      P.run_col[j] = ck;
      P.run_rank[j] = lane;
      P.run_len[j] = (rest ? __ffs(rest) - 1 : nc) - lane;
    }
    if (lane == 0) {
      P.nr = nr;
      P.ncols = nc;
      P.nruns = __popc(sm);
      P.row_bytes = (uint32_t)nc * (16u * kRowsUnits<TMap>);
    }
  }
  if (lane == 0) {
    P.roi = roi;
    P.base = m.base;
    P.W = m.W;
    P.mode = mode;
    if (level_out && src.mode == 0) level_out[roi] = level;
  }
  __syncwarp();
}

// counter[0]: next ROI ticket, counter[1]: CTAs that have drawn their last ticket. Both are zero between launches: the
// last CTA to finish resets them (the workspace is zero-initialised once by its owner).
// Warps 0 .. pw-1 are the consumers (warp = x bin), warp pw the issuer, warp pw+1 the planner.
// `out` is addressed in 16-byte map units (OutUnit): a pixel is kRowsUnits<TMap> of them.
template <typename TMap, typename TOut>
__device__ __forceinline__ void crop_rows_body(const RoiSource& src, int64_t n_rois, int32_t ph, int32_t pw, float extrap,
                                               typename OutUnit<TMap, TOut>::T* __restrict__ out,
                                               int32_t* __restrict__ level_out, unsigned int* __restrict__ counter) {
  using Raw = typename MapUnit<TMap>::Raw;
  using Val = typename MapUnit<TMap>::Val;
  using Out = typename OutUnit<TMap, TOut>::T;
  constexpr int kPixUnits = kRowsUnits<TMap>;             // 64 fp32 quads or 32 bf16 octets
  constexpr int kPixShift = kPixUnits == 64 ? 6 : 5;
  static_assert((1 << kPixShift) == kPixUnits, "a pixel is 64 or 32 units");
  constexpr int kLaneUnits = kPixUnits / 32;              // units per consumer lane and pixel: 8 channels either way
  constexpr uint32_t kPixBytes = 16u * kPixUnits;
  pdl_prologue();
  extern __shared__ __align__(128) unsigned char s_ring[];
  __shared__ RowsShared S;
  const int32_t t = threadIdx.x;
  const int32_t lane = t & 31, warp = t >> 5;
  const int32_t n_cwarps = pw, n_cons = 32 * n_cwarps;
  if (t == 0) {
    for (int32_t e = 0; e < kRowsEntries; ++e) {
      mbar_init(&S.full[e], 1);
      mbar_init(&S.empty[e], (uint32_t)n_cwarps);
    }
    for (int32_t p = 0; p < kRowsPlans; ++p) {
      mbar_init(&S.plan_full[p], 1);
      mbar_init(&S.plan_empty[p], (uint32_t)n_cwarps + 1u);    // consumer warps + the issuer
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncthreads();
  int32_t ps = 0;                                // plan slot + phase, advanced identically by every role
  uint32_t pphase = 0;

  if (warp == n_cwarps + 1) {
    // ------------------------------------------------------------------ planner: draws ROIs, plans a few ahead
    // The ticket is drawn two plans ahead and the box fetched one plan ahead, so that neither the atomic's nor the
    // load's round trip sits between two plans. A CTA therefore draws up to two tickets past the end; the reset of the
    // counters below waits for all of them.
    const int64_t stride = gridDim.x;
    auto draw = [&](int64_t k) -> int64_t {         // k-th ROI of this CTA; dynamic: valid on lane 0 only (see bcast)
      if (!counter) return (int64_t)blockIdx.x + k * stride;
      return lane == 0 ? (int64_t)atomicAdd(&counter[0], 1u) : 0;
    };
    auto bcast = [&](int64_t r) -> int64_t {        // the shuffle is what waits for the atomic: done one plan later
      if (counter) r = (int64_t)__shfl_sync(0xffffffffu, (unsigned int)r, 0);
      if (src.order && r < n_rois) {                                        // ticket -> ROI in processing order
        r = (int64_t)__ldg(&src.order[r]);
        if (r < 0 || r >= n_rois) r = -1;                                   // bad entry of a caller-supplied order: skipped
      }
      return r;
    };
    auto fetch = [&](int64_t r, float4& bx, int32_t& bi) {
      bx = make_float4(0.f, 0.f, 0.f, 0.f);
      bi = 0;
      if (r >= 0 && r < n_rois) {
        bx = __ldg(&src.boxes[r]);
        if (src.mode == 1) bi = __ldg(&src.box_ind[r]);
      }
    };
    int64_t roi = bcast(draw(0)), roi1 = bcast(draw(1));
    float4 box, box1;
    int32_t bi, bi1;
    fetch(roi, box, bi);
    for (int64_t k = 2;; ++k) {
      fetch(roi1, box1, bi1);
      const int64_t roi2_l0 = draw(k);
      mbar_wait(&S.plan_empty[ps], pphase ^ 1u);
      RowsPlan& P = S.plan[ps];
      if (roi >= n_rois) {
        if (lane == 0) {
          P.mode = kRowsDone;
          mbar_arrive(&S.plan_full[ps]);
          if (counter) {
            __threadfence();                                               // ticket draws before the done count
            if (roi2_l0 >= 0 && atomicAdd(&counter[1], 1u) == gridDim.x - 1) { // every CTA has drawn its last ticket
              counter[0] = 0;
              counter[1] = 0;
            }
          }
        }
        return;
      }
      if (roi < 0) {                                 // invalid order entry: an empty plan keeps the roles in step
        if (lane == 0) {
          P.roi = 0;
          P.mode = kRowsSkip;
        }
        __syncwarp();
      } else {
        rows_make_plan<TMap>(src, roi, box, bi, ph, pw, lane, P, S, level_out);
      }
      if (lane == 0) mbar_arrive(&S.plan_full[ps]);
      if (++ps == kRowsPlans) {
        ps = 0;
        pphase ^= 1u;
      }
      roi = roi1;
      box = box1;
      bi = bi1;
      roi1 = bcast(roi2_l0);
    }
  }

  if (warp == n_cwarps) {
    // ------------------------------------------------------------------ issuer: FIFO byte ring
    // Placement is a pure function of the sequence of row sizes (a row that would straddle the end of the ring starts
    // over at offset 0), so the consumers derive every entry's offset themselves instead of reading it back.
    uint32_t head = 0, used = 0;
    int32_t e_idx = 0, old_idx = 0, outstanding = 0;
    uint32_t old_phase = 0;
    const uint64_t pol = l2_policy_evict_normal();
    for (;;) {
      mbar_wait(&S.plan_full[ps], pphase);
      const RowsPlan& P = S.plan[ps];
      const int32_t mode = P.mode;
      if (mode == kRowsDone) return;
      if (mode == kRowsRing) {
        const int32_t nr = P.nr, nruns = P.nruns;
        const uint32_t bytes = P.row_bytes;
        const char* __restrict__ gbase = static_cast<const char*>(P.base);
        const size_t row_pitch = (size_t)P.W * kPixBytes;
        // this lane's column run (nruns <= 16): smem offset inside the row, global offset inside the feature row, bytes
        const int32_t jr = lane < nruns ? lane : 0;
        const uint32_t run_dst = (uint32_t)P.run_rank[jr] * kPixBytes;
        const size_t run_src = (size_t)P.run_col[jr] * kPixBytes;
        const uint32_t run_bytes = (uint32_t)P.run_len[jr] * kPixBytes;
        int32_t my_row = lane < nr ? P.rows[lane] : 0;           // rank k's feature row lives on lane k (nr <= 32)
        for (int32_t k = 0; k < nr; ++k) {
          const bool wrap = head + bytes > kRowsRingBytes;        // the tail a wrapped row skips counts as part of it
          const uint32_t need = bytes + (wrap ? kRowsRingBytes - head : 0u);
          OD_DBG_ASSERT(need <= kRowsRingBytes, "a row and the ring tail it skips exceed the ring");
          while (used + need > kRowsRingBytes || outstanding == kRowsEntries) {
            mbar_wait(&S.empty[old_idx], old_phase);              // reclaim the oldest entry (FIFO)
            used -= S.entry_fp[old_idx];
            --outstanding;
            if (++old_idx == kRowsEntries) {
              old_idx = 0;
              old_phase ^= 1u;
            }
          }
          const uint32_t off = wrap ? 0u : head;
          OD_DBG_ASSERT(off + bytes <= kRowsRingBytes && run_dst + run_bytes <= bytes && bytes > 0, "row outside the ring");
          OD_DBG_IDX(e_idx, kRowsEntries);
          head = off + bytes;
          used += need;
          ++outstanding;
          if (lane == 0) {
            S.entry_fp[e_idx] = need;
            mbar_expect_tx(&S.full[e_idx], bytes);
          }
          __syncwarp();
          const char* srow = gbase + (size_t)__shfl_sync(0xffffffffu, my_row, k) * row_pitch;
          if (lane < nruns) bulk_g2s_hint(s_ring + off + run_dst, srow + run_src, run_bytes, &S.full[e_idx], pol);
          if (++e_idx == kRowsEntries) e_idx = 0;
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&S.plan_empty[ps]);
      if (++ps == kRowsPlans) {
        ps = 0;
        pphase ^= 1u;
      }
    }
  }

  // -------------------------------------------------------------------- consumers
  // warp = x bin, lane = channel quads `lane` and `lane + 32` (fp32 maps) or channel octet `lane` (bf16 maps, one 16-byte
  // LDS per tap pixel): one output pixel per warp and output row.
  const int32_t x = warp;
  const Val ext4 = splat_unit<Val>(extrap);
  int32_t e_idx = 0;
  uint32_t e_phase = 0, c_head = 0;              // ring entry, its phase, and the issuer's head replayed locally
  for (;;) {
    mbar_wait(&S.plan_full[ps], pphase);
    const RowsPlan& P = S.plan[ps];
    const int32_t mode = P.mode;
    if (mode == kRowsDone) break;
    Out* __restrict__ o = out + P.roi * ((int64_t)ph * pw * kPixUnits);
    if (mode == kRowsRing) {
      // Column ranks -> unit index inside a ring row (+ the lane's channel unit).
      const int32_t xcl = P.x_cl[x] * kPixUnits + lane, xcr = P.x_cr[x] * kPixUnits + lane;
      const float xl = P.x_lerp[x];
      const int32_t nr = P.nr;
      const uint32_t row_bytes = P.row_bytes;
      // Rank-major walk: the y's whose top row has rank k are contiguous (P.yfirst), their bottom row is rank k or k+1.
      // Rows alternate between RA (even ranks) and RB (odd ranks). bottom - top is recomputed per y: a group holds 1.2 y's
      // on average, caching the difference would only cost registers.
      Val RA[kLaneUnits], RB[kLaneUnits];
      for (int i = 0; i < kLaneUnits; ++i) RA[i] = RB[i] = ext4;
#define OD_ROWS_LOAD(V)                                                                              \
  do {                                                                                               \
    const uint32_t off_ = (c_head + row_bytes > kRowsRingBytes) ? 0u : c_head;                       \
    c_head = off_ + row_bytes;                                                                       \
    OD_DBG_ASSERT(c_head <= kRowsRingBytes && (uint32_t)(xcr + 32 * (kLaneUnits - 1)) * 16u < row_bytes && xcl <= xcr, \
                  "ring read outside the row");                                                      \
    mbar_wait(&S.full[e_idx], e_phase);                                                              \
    const Raw* rowp = reinterpret_cast<const Raw*>(s_ring + off_);                                   \
    _Pragma("unroll") for (int i = 0; i < kLaneUnits; ++i) {                                         \
      const Val l_ = widen_unit(rowp[xcl + 32 * i]), r_ = widen_unit(rowp[xcr + 32 * i]);            \
      V[i] = axpy4p(l_, sub4p(r_, l_), xl);                                                          \
    }                                                                                                \
    __syncwarp();                                                                                    \
    if (lane == 0) mbar_arrive(&S.empty[e_idx]);                                                     \
    if (++e_idx == kRowsEntries) {                                                                   \
      e_idx = 0;                                                                                     \
      e_phase ^= 1u;                                                                                 \
    }                                                                                                \
  } while (0)
#define OD_ROWS_GROUP(CUR, NXT)                                                                      \
  {                                                                                                  \
    OD_DBG_IDX(k + 1, 2 * kRowsMaxPool + 1);                                                         \
    const int32_t yend = P.yfirst[k + 1];                                                            \
    OD_DBG_ASSERT(yend <= ph && P.roi >= 0 && P.roi < n_rois, "y group / ROI outside the crop");     \
    const bool more = k + 1 < nr;                                                                    \
    if (more) OD_ROWS_LOAD(NXT);                                                                     \
    _Pragma("unroll 1") while (y < yend) {                                                           \
      const int2 nxt_ = P.ytab[y + 2];      /* two rows ahead: the read is off the critical path */    \
      const float yl = __int_as_float(ent.x);                                                        \
      Val v_[kLaneUnits];                                                                            \
      if (ent.y) {                    /* top row == bottom row: (top - top) * yl, as the reference */ \
        _Pragma("unroll") for (int i = 0; i < kLaneUnits; ++i) v_[i] = axpy4p(CUR[i], sub4p(CUR[i], CUR[i]), yl); \
      } else {                                                                                       \
        _Pragma("unroll") for (int i = 0; i < kLaneUnits; ++i) v_[i] = axpy4p(CUR[i], sub4p(NXT[i], CUR[i]), yl); \
      }                                                                                              \
      _Pragma("unroll") for (int i = 0; i < kLaneUnits; ++i) st_unit(orow + lane + 32 * i, v_[i]);   \
      ent = ent1;                                                                                    \
      ent1 = nxt_;                                                                                   \
      ++y;                                                                                           \
      orow += pw * kPixUnits;                                                                        \
    }                                                                                                \
    if (!more) break;                                                                                \
    ++k;                                                                                             \
  }
      Out* __restrict__ orow = o + x * kPixUnits;     // this warp's pixel of output row 0
      int2 ent = P.ytab[0], ent1 = P.ytab[1];
      int32_t y = 0, k = 0;
      OD_ROWS_LOAD(RA);
      for (;;) {
        OD_ROWS_GROUP(RA, RB)
        OD_ROWS_GROUP(RB, RA)
      }
#undef OD_ROWS_LOAD
#undef OD_ROWS_GROUP
    } else if (mode == kRowsFlat) {   // per-bin path: 4 direct loads per output quad
      const Raw* __restrict__ base = static_cast<const Raw*>(P.base);
      const uint32_t W = (uint32_t)P.W;
      const int32_t total = ph * pw * kPixUnits;
      for (int32_t e = t; e < total; e += n_cons) {
        const int32_t bin = e >> kPixShift;
        const uint32_t c = (uint32_t)(e & (kPixUnits - 1));
        const int32_t y = bin / pw, xb = bin - y * pw;
        Val v = ext4;
        if (P.y_ok[y] && P.x_ok[xb]) {
          const uint32_t top = (uint32_t)P.y_top[y], bot = (uint32_t)P.y_bot[y];
          const uint32_t left = (uint32_t)P.x_left[xb], right = (uint32_t)P.x_right[xb];
          const Val tl = ldg_unit(base + ((top * W + left) * kPixUnits + c));
          const Val tr = ldg_unit(base + ((top * W + right) * kPixUnits + c));
          const Val bl = ldg_unit(base + ((bot * W + left) * kPixUnits + c));
          const Val br = ldg_unit(base + ((bot * W + right) * kPixUnits + c));
          const float xl = P.x_lerp[xb];
          v = lerp4p(lerp4p(tl, tr, xl), lerp4p(bl, br, xl), P.y_lerp[y]);
        }
        st_unit(o + e, v);
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&S.plan_empty[ps]);   // this warp no longer reads the plan
    if (++ps == kRowsPlans) {
      ps = 0;
      pphase ^= 1u;
    }
  }
}

__global__ void __launch_bounds__(kRowsThreads, 1)
crop_rows_kernel(RoiSource src, int64_t n_rois, int32_t ph, int32_t pw, float extrap, float4* __restrict__ out,
                 int32_t* __restrict__ level_out, unsigned int* __restrict__ counter) {
  crop_rows_body<float, float>(src, n_rois, ph, pw, extrap, out, level_out, counter);
}
// bf16 maps and / or a bf16 output: the same body, an overload of the same name (the fp32 kernel above keeps its name)
template <typename TMap, typename TOut>
__global__ void __launch_bounds__(kRowsThreads, 1)
crop_rows_kernel(RoiSource src, int64_t n_rois, int32_t ph, int32_t pw, float extrap,
                 typename OutUnit<TMap, TOut>::T* __restrict__ out, int32_t* __restrict__ level_out,
                 unsigned int* __restrict__ counter) {
  crop_rows_body<TMap, TOut>(src, n_rois, ph, pw, extrap, out, level_out, counter);
}

// FasterRCNN roi_pool (fastrcnn.py:22-70): crop_and_resize to (2*oh) x (2*ow) fused with max_pool 2x2 / stride 2.
// Same flat-bin scheme as crop_bins_kernel over the POOLED bins: a CTA owns kPoolBins pooled bins, its table has 4
// entries (the 2x2 sub-bins) per pooled bin; per output quad a thread issues the 16 unconditional 16-byte loads of the
// four sub-bins, blends each and takes the max in the visiting order (0,0),(0,1),(1,0),(1,1). Out-of-range samples
// contribute the extrapolation value 0; a row whose batch index is out of range yields zeros.
constexpr int kPoolBins = 32;
__global__ void __launch_bounds__(kBinThreads)
crop_pool_bins_kernel(RoiSource src, int64_t total_bins, int32_t oh, int32_t ow, int32_t D4, float4* __restrict__ out) {
  __shared__ BinTaps s_taps[kPoolBins * 4];
  __shared__ BinInfo s_info[kPoolBins * 4];
  const int32_t t = threadIdx.x;
  const int64_t bin0 = (int64_t)blockIdx.x * kPoolBins;
  const int32_t nb = (int32_t)min((int64_t)kPoolBins, total_bins - bin0);
  const int32_t bins_per_roi = oh * ow;
  for (int32_t i = t; i < nb * 4; i += kBinThreads) {
    const int64_t fb = bin0 + (i >> 2);
    const int64_t roi = fb / bins_per_roi;
    const int32_t ob = (int32_t)(fb - roi * bins_per_roi);
    const int32_t oy = ob / ow, ox = ob - oy * ow;
    bin_table_entry<float>(src, roi, 2 * oy + ((i >> 1) & 1), 2 * ox + (i & 1), false, 2 * oh, 2 * ow, D4, nullptr, &s_taps[i], &s_info[i]);
  }
  __syncthreads();
  const int32_t total = nb * D4;
  float4* __restrict__ o = out + bin0 * D4;
  const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int32_t e = t; e < total; e += kBinThreads) {
    const int32_t bin = e / D4;
    const uint32_t c = (uint32_t)(e - bin * D4);
    float4 tl[4], tr[4], bl[4], br[4];
    float xl[4], yl[4];
    uint32_t fl[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const BinTaps tp = s_taps[bin * 4 + q];
      const BinInfo bi = s_info[bin * 4 + q];
      const float4* __restrict__ base = reinterpret_cast<const float4*>(bi.base_flag & ~(uintptr_t)15);
      fl[q] = (uint32_t)(bi.base_flag & 3u);
      xl[q] = bi.xl;
      yl[q] = bi.yl;
      tl[q] = ldg_f4(base + (tp.tl + c));
      tr[q] = ldg_f4(base + (tp.tr + c));
      bl[q] = ldg_f4(base + (tp.bl + c));
      br[q] = ldg_f4(base + (tp.br + c));
    }
    float4 v[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float4 top = lerp4p(tl[q], tr[q], xl[q]);
      const float4 bot = lerp4p(bl[q], br[q], xl[q]);
      v[q] = lerp4p(top, bot, yl[q]);
      if (fl[q] != (uint32_t)kBinSample) v[q] = zero4;
    }
    stg_cs_f4(o + e, max4(max4(max4(v[0], v[1]), v[2]), v[3]));
  }
}

// ----------------------------------------------------------------------------- host side
// Shapes crop_rows_kernel serves; every other shape goes to crop_bins_kernel.
static bool crop_rows_serves(const RoiSource& src, int64_t n_rois, int32_t ph, int32_t pw, int32_t D) {
  const int32_t pmax = ph > pw ? ph : pw;
  if (D != 4 * kRowsD4 || ph > kRowsMaxPool || pw > kRowsMaxWidth || pmax < kRowsMinPool || src.mode > 1) return false;
  return n_rois + 4096 <= 0x7FFFFFFFll;
}

// The kernels of one (maps, pooled) dtype pair: the fp32 kernels for fp32 -> fp32, their bf16 overloads otherwise.
template <typename TMap, typename TOut>
constexpr bool kFp32Pair = std::is_same<TMap, float>::value && std::is_same<TOut, float>::value;
template <typename TMap, typename TOut>
static auto rows_kernel() {
  if constexpr (kFp32Pair<TMap, TOut>)
    return static_cast<void (*)(RoiSource, int64_t, int32_t, int32_t, float, float4*, int32_t*, unsigned int*)>(crop_rows_kernel);
  else
    return &crop_rows_kernel<TMap, TOut>;
}
template <typename TMap, typename TOut, int BINS, int UNROLL, bool POW2, bool ORDERED>
static auto bins_kernel() {
  if constexpr (kFp32Pair<TMap, TOut>) return &crop_bins_kernel<BINS, UNROLL, POW2, ORDERED>;
  else return &crop_bins_kernel<TMap, TOut, BINS, UNROLL, POW2, ORDERED>;
}

// returns OD_OK after launching, or 1 when the shape is not served by this kernel (caller falls back to crop_bins).
// `counter`: two zeroed uint32 in the caller's workspace (dynamic ROI scheduling) or NULL (static round robin).
template <typename TMap, typename TOut>
static int launch_crop_rows(const RoiSource& src, int64_t n_rois, int32_t ph, int32_t pw, int32_t D, float extrap, void* out,
                            int32_t* level_out, unsigned int* counter, cudaStream_t st) {
  if (!crop_rows_serves(src, n_rois, ph, pw, D)) return 1;
  static bool configured[64] = {false};    // dynamic shared memory opted in, per device (and dtype pair)
  static int sms[64] = {0};
  const auto kernel = rows_kernel<TMap, TOut>();
  int dev = 0;
  OD_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) OD_FAIL(OD_ERR_DEVICE, "device index %d not supported", dev);
  if (!configured[dev]) {
    OD_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kRowsRingBytes));
    configured[dev] = true;
  }
  if (!sms[dev]) OD_CUDA(cudaDeviceGetAttribute(&sms[dev], cudaDevAttrMultiProcessorCount, dev));
  const int64_t grid = n_rois < (int64_t)sms[dev] ? n_rois : (int64_t)sms[dev];
  OD_CUDA(launch_pdl(kernel, dim3((unsigned)grid), dim3((unsigned)(32 * pw + 64)), (size_t)kRowsRingBytes, st, src,
                     n_rois, ph, pw, extrap, static_cast<typename OutUnit<TMap, TOut>::T*>(out), level_out, counter));
  OD_LAUNCH_CHECK("crop_rows_kernel");
  return OD_OK;
}

static int launch_roi_order(const RoiSource& src, int32_t* order_buf, cudaStream_t st) {
  OD_CUDA(launch_pdl(roi_order_kernel, dim3((unsigned)src.batch), dim3(kOrderThreads), 0, st, src.boxes, src.rois_per_image,
                     src.image_h, src.image_w, src.min_level, src.num_levels, order_buf));
  OD_LAUNCH_CHECK("roi_order_kernel");
  return OD_OK;
}

// `order_buf`: scratch for the pre-pass (or NULL); `order_in`: an order the caller already has (od_roi_processing_order),
// which saves the pre-pass - e.g. the 7x7 and the 14x14 pooling of one step walk the same ROIs.
// D: channels; D4: 16-byte units per pixel.
template <typename TMap, typename TOut>
static int launch_crop_bins(RoiSource src, int64_t n_rois, int32_t ph, int32_t pw, int32_t D, float extrap,
                            void* out, int32_t* level_out, cudaStream_t st, unsigned int* counter = nullptr,
                            int32_t* order_buf = nullptr, const int32_t* order_in = nullptr) {
  using Out = typename OutUnit<TMap, TOut>::T;
  if (n_rois == 0) return OD_OK;
  const int32_t D4 = D / MapUnit<TMap>::kCh;
  // processing order (PyramidROIAlign with a sized workspace, enough ROIs for the order to matter). Measured: +3 % on the
  // persistent 14x14 kernel. For the flat 7x7 kernel the launch itself gets ~2 us faster but its pre-pass adds more than
  // that to a stand-alone call; with several steps in flight (the throughput case) that latency is hidden and the order is
  // worth +2.5 % images/s, so it is on for both (profiles/r2_roialign.md).
  src.order = nullptr;
  const bool order_ok = src.mode == 0 && D == 4 * kRowsD4 && n_rois <= 0x7FFFFFFFll;
  if (order_ok && order_in) {
    src.order = order_in;
  } else if (order_ok && order_buf && n_rois >= 512 && src.rois_per_image <= kOrderThreads * kOrderPerThread) {
    OD_CHECK(launch_roi_order(src, order_buf, st));
    src.order = order_buf;
  }
  const int64_t bins_per_roi = (int64_t)ph * pw;
  if (bins_per_roi > 0x7FFFFFFFll) OD_FAIL(OD_ERR_PARAM, "pool shape %dx%d too large", ph, pw);
  const int64_t total_bins = n_rois * bins_per_roi;
  for (int l = 0; l < (src.mode == 0 ? src.num_levels : 1); ++l)
    if ((int64_t)src.lt.H[l] * src.lt.W[l] * D4 > 0xFFFFFFFFll)
      OD_FAIL(OD_ERR_PARAM, "one image of level %d exceeds 2^32 16-byte units", l);
  {
    const int rc = launch_crop_rows<TMap, TOut>(src, n_rois, ph, pw, D, extrap, out, level_out, counter, st);
    if (rc != 1) return rc;
  }
  int32_t lg = -1;
  if ((D4 & (D4 - 1)) == 0) {
    lg = 0;
    while ((1 << lg) < D4) ++lg;
  }
  // The tier is chosen on 16-byte units per pixel, i.e. on bytes per pixel, not on channels: bf16 maps with D = 64 (8
  // units) take the 512-bin kernel like fp32 maps with D = 32, while fp32 maps with D = 64 (16 units) take the 32-bin one.
  if (lg >= 0 && D4 >= 16) {
    if ((int64_t)64 * D4 > 0x7FFFFFFFll) OD_FAIL(OD_ERR_PARAM, "depth %d too large", D);
    const int64_t grid = (total_bins + kBinBins - 1) / kBinBins;
    if (grid > 0x7FFFFFFFll) OD_FAIL(OD_ERR_PARAM, "too many bins: %lld", (long long)total_bins);
    if (src.order)
      OD_CUDA(launch_pdl(bins_kernel<TMap, TOut, kBinBins, kBinUnroll, true, true>(), dim3((unsigned)grid), dim3(kBinThreads), 0,
          st, src, total_bins, (int32_t)bins_per_roi, ph, pw, D4, lg, extrap, static_cast<Out*>(out), level_out));
    else
      OD_CUDA(launch_pdl(bins_kernel<TMap, TOut, kBinBins, kBinUnroll, true, false>(), dim3((unsigned)grid), dim3(kBinThreads), 0,
          st, src, total_bins, (int32_t)bins_per_roi, ph, pw, D4, lg, extrap, static_cast<Out*>(out), level_out));
  } else {
    // thin or non-power-of-two depth: more bins per CTA so that the table build is amortised
    constexpr int BINS = 512;
    if ((int64_t)BINS * D4 > 0x7FFFFFFFll) OD_FAIL(OD_ERR_PARAM, "depth %d too large", D);
    const int64_t grid = (total_bins + BINS - 1) / BINS;
    if (grid > 0x7FFFFFFFll) OD_FAIL(OD_ERR_PARAM, "too many bins: %lld", (long long)total_bins);
    const auto kernel = lg >= 0 ? bins_kernel<TMap, TOut, BINS, 2, true, false>() : bins_kernel<TMap, TOut, BINS, 2, false, false>();
    kernel<<<(unsigned)grid, kBinThreads, 0, st>>>(src, total_bins, (int32_t)bins_per_roi, ph, pw, D4, lg, extrap,
                                                   static_cast<Out*>(out), level_out);
  }
  OD_LAUNCH_CHECK("crop_bins_kernel");
  return OD_OK;
}

// The dtype a ROIAlign map or output tensor is checked against: BF16 for a bfloat16 tensor, F32 for anything else, which
// check_tensor then refuses unless it is fp32 (float16 included).
static DType map_or_out_dtype(const DLTensor* t) {
  return (t && t->dtype.code == kDLBfloat && t->dtype.bits == 16 && t->dtype.lanes == 1) ? BF16 : F32;
}
// With a bf16 map or output a pixel must be whole 16-byte units of 8 channels.
static int check_bf16_depth(DType map_dt, DType out_dt, int64_t D) {
  if ((map_dt == BF16 || out_dt == BF16) && D % 8)
    OD_FAIL(OD_ERR_SHAPE, "depth %lld must be a multiple of 8 with bfloat16 maps or output", (long long)D);
  return OD_OK;
}
template <typename... Args>
static int launch_crop(DType map_dt, DType out_dt, Args... args) {
  if (map_dt == BF16)
    return out_dt == BF16 ? launch_crop_bins<__nv_bfloat16, __nv_bfloat16>(args...) : launch_crop_bins<__nv_bfloat16, float>(args...);
  return out_dt == BF16 ? launch_crop_bins<float, __nv_bfloat16>(args...) : launch_crop_bins<float, float>(args...);
}

}  // namespace od

using namespace od;

extern "C" {

size_t od_pyramid_roi_align_workspace_bytes(void) { return 256; }
size_t od_pyramid_roi_align_workspace_bytes_n(int64_t n_rois) {
  return 256 + align_up((size_t)(n_rois > 0 ? n_rois : 0) * sizeof(int32_t), 256);
}

int od_roi_processing_order(const DLTensor* rois, int32_t image_h, int32_t image_w, int32_t min_level, int32_t num_levels,
                            DLTensor* order, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  DeviceScope scope;
  OD_CHECK(check_tensor(rois, "rois", F32, {kAny, kAny, 4}, 16, scope));
  const int64_t B = rois->shape[0], N = rois->shape[1];
  OD_CHECK(check_tensor(order, "order", I32, {B * N}, 4, scope));
  if (num_levels < 1 || num_levels > OD_MAX_LEVELS) OD_FAIL(OD_ERR_PARAM, "num_levels %d not in [1,%d]", num_levels, OD_MAX_LEVELS);
  if (B * N == 0) return OD_OK;
  if (B * N > 0x7FFFFFFFll || B > 65535) OD_FAIL(OD_ERR_PARAM, "too many ROIs");
  if (N > kOrderThreads * kOrderPerThread) OD_FAIL(OD_ERR_PARAM, "at most %d ROIs per image", kOrderThreads * kOrderPerThread);
  RoiSource src;
  memset(&src, 0, sizeof(src));
  src.rois_per_image = (int32_t)N;
  src.image_h = image_h;
  src.image_w = image_w;
  src.min_level = min_level;
  src.num_levels = num_levels;
  src.batch = (int32_t)B;
  src.boxes = dptr<float4>(rois);
  return launch_roi_order(src, dptr<int32_t>(order), st);
}

int od_pyramid_roi_align_forward_ws(const DLTensor* const* fmaps, int32_t num_levels, int32_t min_level,
                                    const DLTensor* rois, int32_t image_h, int32_t image_w, int32_t pool_h,
                                    int32_t pool_w, DLTensor* pooled, DLTensor* roi_level, void* ws, size_t ws_bytes,
                                    void* stream) {
  return od_pyramid_roi_align_forward_ordered(fmaps, num_levels, min_level, rois, image_h, image_w, pool_h, pool_w, pooled,
                                              roi_level, nullptr, ws, ws_bytes, stream);
}

int od_pyramid_roi_align_forward_ordered(const DLTensor* const* fmaps, int32_t num_levels, int32_t min_level,
                                         const DLTensor* rois, int32_t image_h, int32_t image_w, int32_t pool_h,
                                         int32_t pool_w, DLTensor* pooled, DLTensor* roi_level, const DLTensor* order,
                                         void* ws, size_t ws_bytes, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (!fmaps) OD_FAIL(OD_ERR_NULL, "fmaps is NULL");
  if (num_levels < 1 || num_levels > OD_MAX_LEVELS) OD_FAIL(OD_ERR_PARAM, "num_levels %d not in [1,%d]", num_levels, OD_MAX_LEVELS);
  if (pool_h < 1 || pool_w < 1) OD_FAIL(OD_ERR_PARAM, "pool shape %dx%d unsupported", pool_h, pool_w);
  DeviceScope scope;
  OD_CHECK(check_tensor(rois, "rois", F32, {kAny, kAny, 4}, 16, scope));
  const int64_t B = rois->shape[0], N = rois->shape[1];
  LevelTable lt;
  int64_t D = kAny;   // that of the first level
  const DType map_dt = map_or_out_dtype(fmaps[0]);   // every level must have the first level's dtype
  for (int l = 0; l < num_levels; ++l) {
    OD_CHECK(check_tensor(fmaps[l], "fmaps[l]", map_dt, {B, kAny, kAny, D}, 16, scope));
    D = fmaps[l]->shape[3];
    lt.ptr[l] = dptr<char>(fmaps[l]);
    lt.H[l] = (int32_t)fmaps[l]->shape[1];
    lt.W[l] = (int32_t)fmaps[l]->shape[2];
  }
  if (D % 4) OD_FAIL(OD_ERR_SHAPE, "depth %lld must be a multiple of 4", (long long)D);
  const DType out_dt = map_or_out_dtype(pooled);
  if (pooled && pooled->ndim == 5) OD_CHECK(check_tensor(pooled, "pooled", out_dt, {1, B * N, pool_h, pool_w, D}, 16, scope));
  else OD_CHECK(check_tensor(pooled, "pooled", out_dt, {B * N, pool_h, pool_w, D}, 16, scope));
  OD_CHECK(check_bf16_depth(map_dt, out_dt, D));
  OD_CHECK(check_opt_tensor(roi_level, "roi_level", I32, {B, N}, 4, scope));
  const int64_t total = B * N;
  if (total == 0) return OD_OK;
  RoiSource src;
  memset(&src, 0, sizeof(src));
  src.mode = 0;
  src.rois_per_image = (int32_t)N;
  src.image_h = image_h;
  src.image_w = image_w;
  src.min_level = min_level;
  src.num_levels = num_levels;
  src.batch = (int32_t)B;
  src.lt = lt;
  src.boxes = dptr<float4>(rois);
  if (ws && (ws_bytes < od_pyramid_roi_align_workspace_bytes() || reinterpret_cast<uintptr_t>(ws) % 8))
    OD_FAIL(OD_ERR_WORKSPACE, "workspace must be 8-byte aligned and at least %zu bytes", od_pyramid_roi_align_workspace_bytes());
  // workspace: [0,256) the ticket counters (stay zeroed), [256, 256 + 4*B*N) the ROI processing order (scratch)
  int32_t* order_buf = (ws && ws_bytes >= od_pyramid_roi_align_workspace_bytes_n(total))
                           ? reinterpret_cast<int32_t*>(static_cast<char*>(ws) + 256) : nullptr;
  OD_CHECK(check_opt_tensor(order, "order", I32, {total}, 4, scope));
  return launch_crop(map_dt, out_dt, src, total, pool_h, pool_w, (int32_t)D, 0.0f, dptr<void>(pooled), dptr<int32_t>(roi_level),
                     st, static_cast<unsigned int*>(ws), order_buf, dptr<int32_t>(order));
}

int od_pyramid_roi_align_forward(const DLTensor* const* fmaps, int32_t num_levels, int32_t min_level,
                                 const DLTensor* rois, int32_t image_h, int32_t image_w, int32_t pool_h,
                                 int32_t pool_w, DLTensor* pooled, DLTensor* roi_level, void* stream) {
  return od_pyramid_roi_align_forward_ws(fmaps, num_levels, min_level, rois, image_h, image_w, pool_h, pool_w, pooled,
                                         roi_level, nullptr, 0, stream);
}


int od_crop_and_resize(const DLTensor* image, const DLTensor* boxes, const DLTensor* box_ind, int32_t crop_h,
                       int32_t crop_w, float extrapolation_value, DLTensor* out, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  DeviceScope scope;
  const DType map_dt = map_or_out_dtype(image), out_dt = map_or_out_dtype(out);
  OD_CHECK(check_tensor(image, "image", map_dt, {kAny, kAny, kAny, kAny}, 16, scope));
  OD_CHECK(check_tensor(boxes, "boxes", F32, {kAny, 4}, 16, scope));
  const int64_t n = boxes->shape[0], D = image->shape[3];
  OD_CHECK(check_tensor(box_ind, "box_ind", I32, {n}, 4, scope));
  if (crop_h < 1 || crop_w < 1) OD_FAIL(OD_ERR_PARAM, "crop size %dx%d unsupported", crop_h, crop_w);
  OD_CHECK(check_tensor(out, "out", out_dt, {n, crop_h, crop_w, D}, 16, scope));
  if (D % 4) OD_FAIL(OD_ERR_SHAPE, "depth %lld must be a multiple of 4", (long long)D);
  OD_CHECK(check_bf16_depth(map_dt, out_dt, D));
  if (n == 0) return OD_OK;
  RoiSource src;
  memset(&src, 0, sizeof(src));
  src.mode = 1;
  src.batch = (int32_t)image->shape[0];
  src.lt.ptr[0] = dptr<char>(image);
  src.lt.H[0] = (int32_t)image->shape[1];
  src.lt.W[0] = (int32_t)image->shape[2];
  src.boxes = dptr<float4>(boxes);
  src.box_ind = dptr<int32_t>(box_ind);
  return launch_crop(map_dt, out_dt, src, n, crop_h, crop_w, (int32_t)D, extrapolation_value, dptr<void>(out), nullptr, st);
}

int od_roi_pool_forward(const DLTensor* feature_map, const DLTensor* proposals, float image_h, float image_w,
                        DLTensor* out, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  DeviceScope scope;
  OD_CHECK(check_tensor(feature_map, "feature_map", F32, {kAny, kAny, kAny, kAny}, 16, scope));
  OD_CHECK(check_tensor(proposals, "proposals", F32, {kAny, 5}, 4, scope));
  const int64_t n = proposals->shape[0], D = feature_map->shape[3];
  OD_CHECK(check_tensor(out, "out", F32, {n, 7, 7, D}, 16, scope));
  if (D % 4) OD_FAIL(OD_ERR_SHAPE, "depth %lld must be a multiple of 4", (long long)D);
  if (n == 0) return OD_OK;
  if ((int64_t)feature_map->shape[1] * feature_map->shape[2] * (D / 4) > 0xFFFFFFFFll)
    OD_FAIL(OD_ERR_PARAM, "feature map exceeds 2^32 16-byte units per image");
  RoiSource src;
  memset(&src, 0, sizeof(src));
  src.mode = 2;
  src.batch = (int32_t)feature_map->shape[0];
  src.lt.ptr[0] = dptr<char>(feature_map);
  src.lt.H[0] = (int32_t)feature_map->shape[1];
  src.lt.W[0] = (int32_t)feature_map->shape[2];
  src.boxes5 = dptr<float>(proposals);
  src.fimage_h = image_h;
  src.fimage_w = image_w;
  const int64_t total_bins = n * 49;
  const int64_t grid = (total_bins + kPoolBins - 1) / kPoolBins;
  if (grid > 0x7FFFFFFFll) OD_FAIL(OD_ERR_PARAM, "too many ROIs");
  crop_pool_bins_kernel<<<(unsigned)grid, kBinThreads, 0, st>>>(src, total_bins, 7, 7, (int32_t)(D / 4), dptr<float4>(out));
  OD_LAUNCH_CHECK("crop_pool_bins_kernel");
  return OD_OK;
}

}  // extern "C"
