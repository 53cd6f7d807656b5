// core.cu — status strings, thread-local error detail, DLPack tensor validation.
#include "common.cuh"

namespace od {

static thread_local char g_detail[512] = "";
static unsigned long long g_launches = 0;

void count_launches(int n) { __atomic_fetch_add(&g_launches, (unsigned long long)n, __ATOMIC_RELAXED); }

void set_error_detail(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_detail, sizeof(g_detail), fmt, ap);
  va_end(ap);
}

static bool is_contiguous(const DLTensor* t) {
  if (!t->strides) return true;
  for (int i = 0; i < t->ndim; ++i)
    if (t->shape[i] == 0) return true;   // no element to address: any strides describe it (torch gives [B,0,4] stride 4)
  int64_t expect = 1;
  for (int i = t->ndim - 1; i >= 0; --i) {
    if (t->shape[i] != 1 && t->strides[i] != expect) return false;
    expect *= t->shape[i];
  }
  return true;
}

int check_tensor(const DLTensor* t, const char* name, DType dt, const int64_t* extents, int ndim, int align_bytes,
                 DeviceScope& scope, bool any_strides) {
  if (!t) OD_FAIL(OD_ERR_NULL, "%s is NULL", name);
  if (t->device.device_type != kDLCUDA)
    OD_FAIL(OD_ERR_DEVICE, "%s: device_type %d is not kDLCUDA (there is no CPU path)", name, (int)t->device.device_type);
  if (scope.device < 0) {
    scope.device = t->device.device_id;
    if (cudaGetDevice(&scope.prev) == cudaSuccess && scope.prev != scope.device && cudaSetDevice(scope.device) == cudaSuccess)
      scope.switched = true;
  } else if (scope.device != t->device.device_id) {
    OD_FAIL(OD_ERR_DEVICE, "%s is on cuda:%d, expected cuda:%d", name, t->device.device_id, scope.device);
  }
  const uint8_t code = (dt == I32) ? (uint8_t)kDLInt : (dt == BF16) ? (uint8_t)kDLBfloat : (uint8_t)kDLFloat;
  const uint8_t bits = (dt == F64) ? 64 : (dt == BF16) ? 16 : 32;
  if (t->dtype.code != code || t->dtype.bits != bits || t->dtype.lanes != 1)
    OD_FAIL(OD_ERR_DTYPE, "%s: dtype (code %d, bits %d) != expected (code %d, bits %d)", name, t->dtype.code,
            t->dtype.bits, code, bits);
  if (ndim >= 0 && t->ndim != ndim) OD_FAIL(OD_ERR_SHAPE, "%s: rank %d != %d", name, t->ndim, ndim);
  for (int i = 0; i < t->ndim; ++i)
    if (t->shape[i] < 0) OD_FAIL(OD_ERR_SHAPE, "%s: negative extent", name);
  if (!any_strides && !is_contiguous(t)) OD_FAIL(OD_ERR_LAYOUT, "%s must be C-contiguous", name);
  const bool empty = numel(t) == 0;
  if (!empty && dptr<char>(t) == nullptr) OD_FAIL(OD_ERR_NULL, "%s: data pointer is NULL", name);
  for (int i = 0; i < ndim; ++i)
    if (extents[i] != kAny && t->shape[i] != extents[i])
      OD_FAIL(OD_ERR_SHAPE, "%s: extent %d is %lld, expected %lld", name, i, (long long)t->shape[i], (long long)extents[i]);
  if (!empty && reinterpret_cast<uintptr_t>(dptr<char>(t)) % align_bytes)
    OD_FAIL(OD_ERR_LAYOUT, "%s is not %d-byte aligned", name, align_bytes);
  return OD_OK;
}

}  // namespace od

extern "C" {

#ifndef OD_SOURCE_HASH
#define OD_SOURCE_HASH "unknown"
#endif
const char* od_source_hash(void) { return OD_SOURCE_HASH; }

int od_version(void) { return 10000 * 0 + 100 * 1 + 0; }

const char* od_strerror(int status) {
  switch (status) {
    case OD_OK: return "ok";
    case OD_ERR_NULL: return "required pointer is NULL";
    case OD_ERR_DTYPE: return "wrong dtype";
    case OD_ERR_SHAPE: return "wrong shape";
    case OD_ERR_DEVICE: return "wrong device (CUDA tensors on one device required)";
    case OD_ERR_LAYOUT: return "tensor must be contiguous / aligned";
    case OD_ERR_WORKSPACE: return "workspace missing or too small";
    case OD_ERR_CUDA: return "CUDA runtime error";
    case OD_ERR_PARAM: return "parameter out of supported range";
    default: return "unknown status";
  }
}

const char* od_last_error_detail(void) { return od::g_detail; }

int64_t od_launch_count(void) { return (int64_t)__atomic_load_n(&od::g_launches, __ATOMIC_RELAXED); }

}  // extern "C"
