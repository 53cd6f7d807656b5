// common.cuh — shared host/device helpers of libodhead.so (sm_100a only).
//
// Numeric contract shared with oracle/odhead_oracle.c so that integer outputs are bit-exact:
//   * fp32 arithmetic in the reference's operation order; the library is compiled with
//     -fmad=false (no FMA contraction), IEEE division and sqrt (nvcc defaults, no fast-math);
//   * exp/log are the correctly rounded fp32 values (evaluated in fp64, then rounded);
//   * min/max are std::min/std::max forms `(b<a)?b:a` / `(a<b)?b:a` (a NaN first operand propagates);
//   * float -> int32 follows x86 cvttss2si (NaN / out of range -> INT_MIN);
//   * ordering ties go to the lower index (composite 64-bit keys).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <string.h>
#include <initializer_list>

#include "../../include/odhead.h"

#ifndef __CUDA_ARCH__
#define OD_HD __host__ __device__
#else
#define OD_HD __host__ __device__
#endif

namespace od {

// ----------------------------------------------------------------------------- errors
void set_error_detail(const char* fmt, ...);
#define OD_FAIL(code, ...)                 \
  do {                                     \
    od::set_error_detail(__VA_ARGS__);     \
    return (code);                         \
  } while (0)
#define OD_CHECK(expr)                     \
  do {                                     \
    int _st = (expr);                      \
    if (_st != OD_OK) return _st;          \
  } while (0)
#define OD_CUDA(expr)                                                                         \
  do {                                                                                        \
    cudaError_t _e = (expr);                                                                  \
    if (_e != cudaSuccess) OD_FAIL(OD_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(_e));     \
  } while (0)
// Kernel-launch statistics (od_launch_count): one relaxed atomic add per launch, no other global state.
void count_launches(int n);
#define OD_LAUNCH_CHECK_NC(name)                                                              \
  do {                                                                                        \
    cudaError_t _e = cudaGetLastError();                                                      \
    if (_e != cudaSuccess) OD_FAIL(OD_ERR_CUDA, "launch %s: %s", name, cudaGetErrorString(_e)); \
  } while (0)
// after exactly ONE kernel launch (loops of launches call count_launches themselves + OD_LAUNCH_CHECK_NC)
#define OD_LAUNCH_CHECK(name)                                                                 \
  do {                                                                                        \
    od::count_launches(1);                                                                    \
    OD_LAUNCH_CHECK_NC(name);                                                                 \
  } while (0)

// ----------------------------------------------------------------------------- device selection
// Every entry point declares one DeviceScope and passes it to check_tensor() for each of its tensors. The first tensor
// checked selects the device: if that is not the calling thread's current device, the scope switches to it (kernel
// launches, cudaFuncSetAttribute and cooperative-launch queries then address the tensors' GPU), every later tensor
// must be on it, and the destructor restores the caller's device.
struct DeviceScope {
  int device = -1;
  int prev = -1;
  bool switched = false;
  ~DeviceScope() {
    if (switched) cudaSetDevice(prev);
  }
};

// ----------------------------------------------------------------------------- DLPack checks
// BF16: kDLBfloat, 16 bits (float16 is kDLFloat, 16 bits, and matches none); U8: kDLUInt, 8 bits; BOOL: kDLBool, 8 bits
enum DType { F32, F64, I32, BF16, U8, BOOL };
// An extent check_tensor accepts at any value. A caller's int64 parameter is checked for a negative value before it is
// used as an extent, so that it cannot pass as kAny.
constexpr int64_t kAny = INT64_MIN;
// Validates one tensor argument, in this order: not NULL, a kDLCUDA tensor on the call's device (see DeviceScope), dtype
// `dt`, rank ndim, no negative extent, C-contiguous (any_strides: any strides), a data pointer unless it is empty,
// extent i == extents[i] (kAny: any value), and, unless it is empty, a data pointer aligned to align_bytes: the size of
// the type the kernels read it as (16 for float4, 8 for float2 and double, else 4). ndim < 0 checks neither rank nor
// extents.
int check_tensor(const DLTensor* t, const char* name, DType dt, const int64_t* extents, int ndim, int align_bytes,
                 DeviceScope& scope, bool any_strides = false);
inline int check_tensor(const DLTensor* t, const char* name, DType dt, std::initializer_list<int64_t> extents,
                        int align_bytes, DeviceScope& scope, bool any_strides = false) {
  return check_tensor(t, name, dt, extents.begin(), (int)extents.size(), align_bytes, scope, any_strides);
}
// The same for an optional argument: NULL is accepted.
inline int check_opt_tensor(const DLTensor* t, const char* name, DType dt, std::initializer_list<int64_t> extents,
                            int align_bytes, DeviceScope& scope) {
  return t ? check_tensor(t, name, dt, extents, align_bytes, scope) : OD_OK;
}
// The dtype an argument that may be fp32 or bf16 is checked against: BF16 for a bfloat16 tensor, F32 for anything else,
// which check_tensor then refuses unless it is fp32 (float16 included). NULL gives F32.
inline DType f32_or_bf16(const DLTensor* t) {
  return (t && t->dtype.code == kDLBfloat && t->dtype.bits == 16 && t->dtype.lanes == 1) ? BF16 : F32;
}
// The same for an argument that may be fp32 or a byte mask (uint8 or bool): U8 or BOOL for an 8-bit kDLUInt or kDLBool
// tensor, F32 for anything else (int8 is kDLInt and is refused). NULL gives F32.
inline DType f32_or_byte(const DLTensor* t) {
  if (!t || t->dtype.bits != 8 || t->dtype.lanes != 1) return F32;
  return t->dtype.code == kDLUInt ? U8 : t->dtype.code == kDLBool ? BOOL : F32;
}
inline int64_t numel(const DLTensor* t) {
  int64_t n = 1;
  for (int i = 0; i < t->ndim; ++i) n *= t->shape[i];
  return n;
}
template <typename T>
inline T* dptr(const DLTensor* t) {
  return t ? reinterpret_cast<T*>(static_cast<char*>(t->data) + t->byte_offset) : nullptr;
}
inline int64_t stride_of(const DLTensor* t, int dim) {
  if (t->strides) return t->strides[dim];
  int64_t s = 1;
  for (int i = t->ndim - 1; i > dim; --i) s *= t->shape[i];
  return s;
}
inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Bump allocator over the caller's workspace.
struct Workspace {
  char* base;
  size_t size;
  size_t off;
  bool dry;  // size query only
  Workspace(void* p, size_t n) : base(static_cast<char*>(p)), size(n), off(0), dry(p == nullptr) {}
  template <typename T>
  T* take(size_t count) {
    off = align_up(off, 256);
    T* p = dry ? nullptr : reinterpret_cast<T*>(base + off);
    off += count * sizeof(T);
    return p;
  }
  bool ok() const { return dry || off <= size; }
};

// ----------------------------------------------------------------------------- debug bounds build
// compute-sanitizer is not available on the GPU pool, so the index-heavy kernels carry their own checks: a library
// built with -DOD_DEBUG_BOUNDS (build.build_variant("dbg", ["OD_DEBUG_BOUNDS"]), selected with ODHEAD_LIB) verifies
// every data-dependent index into shared-memory tables, rings, bitmaps and workspace arrays and traps (with a printf
// naming the site) on the first violation; the -m gpu suite is run against it once per round (profiles/). In the
// product build the macros expand to nothing.
#ifdef OD_DEBUG_BOUNDS
#define OD_DBG_ASSERT(cond, what)                                                                              \
  do {                                                                                                         \
    if (!(cond)) {                                                                                             \
      printf("OD_DEBUG_BOUNDS %s:%d: %s  [block (%d,%d,%d) thread %d]\n", __FILE__, __LINE__, what, (int)blockIdx.x, \
             (int)blockIdx.y, (int)blockIdx.z, (int)threadIdx.x);                                              \
      __trap();                                                                                                \
    }                                                                                                          \
  } while (0)
#else
#define OD_DBG_ASSERT(cond, what) \
  do {                            \
  } while (0)
#endif
#define OD_DBG_IDX(i, n) OD_DBG_ASSERT((long long)(i) >= 0 && (long long)(i) < (long long)(n), #i " in [0, " #n ")")

// ----------------------------------------------------------------------------- programmatic dependent launch
// The proposal front is a chain of ~12 short kernels. Launched with programmatic stream serialisation, the CTAs of kernel
// N+1 become resident while kernel N still runs and block in griddepcontrol.wait until N has completed and flushed, so
// the launch latency of every link overlaps its predecessor. Every kernel on the chain calls pdl_prologue() first, on
// every path (a kernel that finished without waiting would release its own dependents too early). Without the launch
// attribute both instructions are no-ops.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_prologue() {
  pdl_launch_dependents();
  pdl_wait();
}
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ----------------------------------------------------------------------------- exact math
__device__ __forceinline__ float f_min(float a, float b) { return (b < a) ? b : a; }
__device__ __forceinline__ float f_max(float a, float b) { return (a < b) ? b : a; }
__device__ __forceinline__ float f_exp(float x) { return (float)exp((double)x); }
__device__ __forceinline__ float f_log(float x) { return (float)log((double)x); }
__device__ __forceinline__ int32_t f_to_i32_x86(float r) {
  if (!(r > -2147483904.0f && r < 2147483648.0f)) return INT32_MIN;
  return (int32_t)r;
}

// Order-preserving float -> uint32 (larger float = larger key); -0 == +0. Every NaN, of either sign and any payload,
// is one value above +inf (numpy's sort order), so NaN ties go to the lower index like any other tie.
__device__ __forceinline__ uint32_t score_key(float s) {
  if (s != s) return 0xFFFFFFFFu;
  s = s + 0.0f;
  uint32_t b = __float_as_uint(s);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float key_to_score(uint32_t k) {
  uint32_t b = (k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k;
  return __uint_as_float(b);
}
// (score desc, index asc) == composite desc
__device__ __forceinline__ uint64_t composite_key(float s, uint32_t idx) {
  return ((uint64_t)score_key(s) << 32) | (uint64_t)(0xFFFFFFFFu - idx);
}
__device__ __forceinline__ uint32_t composite_index(uint64_t c) { return 0xFFFFFFFFu - (uint32_t)(c & 0xFFFFFFFFull); }

// apply_box_deltas, proposals_tf.py:46-61
__device__ __forceinline__ float4 decode_box(float4 a, float4 d) {
  float height = a.z - a.x;
  float width = a.w - a.y;
  float center_y = a.x + 0.5f * height;
  float center_x = a.y + 0.5f * width;
  center_y = center_y + d.x * height;
  center_x = center_x + d.y * width;
  height = height * f_exp(d.z);
  width = width * f_exp(d.w);
  float y1 = center_y - 0.5f * height;
  float x1 = center_x - 0.5f * width;
  float y2 = y1 + height;
  float x2 = x1 + width;
  return make_float4(y1, x1, y2, x2);
}
// clip_boxes_to_01, proposals_tf.py:86-94; w = (wy1,wx1,wy2,wx2)
__device__ __forceinline__ float4 clip_box(float4 b, float4 w) {
  return make_float4(f_max(f_min(b.x, w.z), w.x), f_max(f_min(b.y, w.w), w.y),
                     f_max(f_min(b.z, w.z), w.x), f_max(f_min(b.w, w.w), w.y));
}

// TF non_max_suppression_op.cc IOU, split into a per-box canonical form + pair test.
struct CBox {  // canonicalised corners + area
  float ymin, xmin, ymax, xmax, area;
};
__device__ __forceinline__ CBox canon_box(float4 b) {
  CBox c;
  c.ymin = f_min(b.x, b.z);
  c.xmin = f_min(b.y, b.w);
  c.ymax = f_max(b.x, b.z);
  c.xmax = f_max(b.y, b.w);
  c.area = (c.ymax - c.ymin) * (c.xmax - c.xmin);
  return c;
}
__device__ __forceinline__ float tf_iou(const CBox& i, const CBox& j) {
  if (i.area <= 0 || j.area <= 0) return 0.0f;
  const float iymin = f_max(i.ymin, j.ymin), ixmin = f_max(i.xmin, j.xmin);
  const float iymax = f_min(i.ymax, j.ymax), ixmax = f_min(i.xmax, j.xmax);
  const float inter = f_max(iymax - iymin, 0.0f) * f_max(ixmax - ixmin, 0.0f);
  return inter / (i.area + j.area - inter);
}

// 16-byte global accesses with cache hints.
__device__ __forceinline__ float4 ldg_f4(const float4* p) { return __ldg(p); }
__device__ __forceinline__ void stg_cs_f4(float4* p, float4 v) { __stcs(p, v); }   // streaming store (evict first)

// Network-head outputs (RPN logits and deltas, classifier probabilities and boxes, the loss inputs) are read as fp32 or
// bf16. A bf16 is the upper half of an fp32, so it is widened exactly with a shift: sign, NaN payload and subnormals
// survive (the library is built without flush-to-zero), and everything after the load is the fp32 path on the widened
// values. Element 0 of a packed pair sits in the low half. Loaded in one access each: one scalar, the i-th (x, y) pair
// (8 B, or 4 B in bf16) or the i-th 4-value row (16 B, or 8 B in bf16) of p.
__device__ __forceinline__ float widen_bf16(uint32_t bits) { return __uint_as_float(bits << 16); }
__device__ __forceinline__ float2 widen_bf16x2(uint32_t u) { return make_float2(widen_bf16(u), __uint_as_float(u & 0xFFFF0000u)); }
__device__ __forceinline__ float ld_head(const float* p) { return *p; }
__device__ __forceinline__ float ld_head(const __nv_bfloat16* p) {
  return widen_bf16(*reinterpret_cast<const unsigned short*>(p));
}
__device__ __forceinline__ float2 ldg_head2(const float* p, int64_t i) { return __ldg(reinterpret_cast<const float2*>(p) + i); }
__device__ __forceinline__ float2 ldg_head2(const __nv_bfloat16* p, int64_t i) {
  return widen_bf16x2(__ldg(reinterpret_cast<const unsigned int*>(p) + i));
}
__device__ __forceinline__ float4 ldg_head4(const float* p, int64_t i) { return __ldg(reinterpret_cast<const float4*>(p) + i); }
__device__ __forceinline__ float4 ldg_head4(const __nv_bfloat16* p, int64_t i) {
  const uint2 u = __ldg(reinterpret_cast<const uint2*>(p) + i);
  const float2 lo = widen_bf16x2(u.x), hi = widen_bf16x2(u.y);
  return make_float4(lo.x, lo.y, hi.x, hi.y);
}

constexpr int kNumSMsB200 = 148;

// A launch gets 48 KiB of shared memory, static and dynamic together, unless its kernel was opted in to more dynamic shared
// memory. The opt-in is needed as soon as the dynamic bytes plus the kernel's static shared memory pass 48 KiB, not only
// when the dynamic bytes alone do. Call sites read the static size once: `static const size_t s = static_smem_bytes(k);`.
inline size_t static_smem_bytes(const void* kernel) {
  cudaFuncAttributes a;
  return cudaFuncGetAttributes(&a, kernel) == cudaSuccess ? a.sharedSizeBytes : (size_t)48 * 1024;   // unknown: opt in
}

}  // namespace od
