// Library-level entry points, error plumbing, TMA descriptor construction.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <atomic>
#include "internal.h"

namespace sres {

static thread_local char t_err[512] = "";

int set_error(int code, const char* msg) {
  snprintf(t_err, sizeof(t_err), "%s", msg ? msg : "");
  return code;
}
int set_cuda_error(cudaError_t e, const char* where) {
  snprintf(t_err, sizeof(t_err), "%s: %s (%s)", where, cudaGetErrorString(e), cudaGetErrorName(e));
  return SRES_ERR_CUDA;
}

int pdl_level() {
  // function-local static with an initialiser: thread-safe one-time read (autograd runs backward on its own thread)
  static const int v = [] {
    const char* e = getenv("SRES_PDL");
    return e ? atoi(e) : 2;  // 2: tensor-core kernels and the channel-attention kernels (measured 29.1 vs 29.5 ms per step)
  }();
  return v;
}
bool pdl_enabled() { return pdl_level() >= 1; }

int device_sm_count() {
  static thread_local int cached_dev = -1, cached_sms = 0;
  int dev = -1;
  if (cudaGetDevice(&dev) != cudaSuccess) {
    cudaGetLastError();
    return -1;
  }
  if (dev != cached_dev) {
    int sms = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) {
      cudaGetLastError();
      return -1;
    }
    cached_dev = dev;
    cached_sms = sms;
  }
  return cached_sms;
}

// Grid of a persistent kernel that walks n_tiles equal tiles: every SM, even when fewer CTAs would finish in the same number
// of waves (1201 tiles take 9 waves on 148 or on 134 CTAs).  With 148 CTAs the 131 that own only 8 tiles free their SMs a
// tile early, and the next kernel's prologue (barriers, TMEM, 72 KB of weights) runs there under programmatic dependent
// launch: the smallest grid measured 1.3 % slower per training step on one B200 (28.49 vs 28.11 ms).
int persistent_grid(int n_tiles, int sms) { return n_tiles < sms ? n_tiles : sms; }

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
    else
      cudaGetLastError();
  }
  return fn;
}

int make_tmap_rows64(CUtensorMap* out, const void* base, uint64_t nrows, uint32_t box_rows) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return set_error(SRES_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
  if ((reinterpret_cast<uintptr_t>(base) & 127) != 0)
    return set_error(SRES_ERR_INVALID_ARG, "TMA operand must be 128-byte aligned");
  cuuint64_t dims[2] = {64, nrows};
  cuuint64_t strides[1] = {128};
  cuuint32_t box[2] = {64, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char msg[128];
    snprintf(msg, sizeof(msg), "cuTensorMapEncodeTiled failed (CUresult %d, rows %llu, box %u)", (int)r,
             (unsigned long long)nrows, box_rows);
    return set_error(SRES_ERR_CUDA, msg);
  }
  return SRES_OK;
}

int make_tmap_rows64_f32(CUtensorMap* out, const void* base, uint64_t nrows, uint32_t box_rows) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return set_error(SRES_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
  if ((reinterpret_cast<uintptr_t>(base) & 127) != 0)
    return set_error(SRES_ERR_INVALID_ARG, "TMA operand must be 128-byte aligned");
  cuuint64_t dims[2] = {64, nrows};
  cuuint64_t strides[1] = {256};
  cuuint32_t box[2] = {32, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error(SRES_ERR_CUDA, "cuTensorMapEncodeTiled (fp32) failed");
  return SRES_OK;
}

int make_tmap_rows64_half(CUtensorMap* out, const void* base, uint64_t nrows, uint32_t box_rows) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return set_error(SRES_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
  if ((reinterpret_cast<uintptr_t>(base) & 127) != 0)
    return set_error(SRES_ERR_INVALID_ARG, "TMA operand must be 128-byte aligned");
  cuuint64_t dims[2] = {64, nrows};
  cuuint64_t strides[1] = {128};
  cuuint32_t box[2] = {32, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_error(SRES_ERR_CUDA, "cuTensorMapEncodeTiled (bf16 half rows) failed");
  return SRES_OK;
}

}  // namespace sres

namespace sres {
static std::atomic<long long> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
}  // namespace sres
extern "C" long long sres_launch_count(void) { return sres::g_launches.load(std::memory_order_relaxed); }
extern "C" int sres_abi_version(void) { return 4; }  // 4: image-resident RCAB chain and split-trunk channel-attention entry points removed
extern "C" const char* sres_last_error(void) { return sres::t_err; }
extern "C" int sres_device_sm_count(void) { return sres::device_sm_count(); }
extern "C" int64_t sres_ptl_rows(int B, int H, int W) { return (int64_t)B * (H + 1) * (W + 1); }

// ---------------------------------------------------------------------------------------------
// L2 residency hints: keep the fp32 residual / gradient trunk (read-modify-written by every RCAB)
// in the persisting part of L2 so that it never round-trips through HBM.
// ---------------------------------------------------------------------------------------------
namespace sres {
// Set by sres_l2_set_aside(bytes > 0) for the device that was current at the call; the executors mark the trunks persisting on
// that device only (the set-aside is a per-device CUDA limit).  -1 = never requested.
static std::atomic<int> g_l2_hint_device{-1};
bool l2_hint_enabled() {
  const int want = g_l2_hint_device.load(std::memory_order_relaxed);
  if (want < 0) return false;
  int dev = -1;
  return cudaGetDevice(&dev) == cudaSuccess && dev == want;
}
}  // namespace sres

extern "C" int sres_l2_set_aside(size_t bytes) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return sres::set_cuda_error(e, "l2_set_aside: device");
  int max_bytes = 0;
  cudaDeviceGetAttribute(&max_bytes, cudaDevAttrMaxPersistingL2CacheSize, dev);
  if (bytes > (size_t)max_bytes) bytes = (size_t)max_bytes;
  e = cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, bytes);
  if (e != cudaSuccess) return sres::set_cuda_error(e, "l2_set_aside: cudaDeviceSetLimit");
  sres::g_l2_hint_device.store(bytes > 0 ? dev : -1, std::memory_order_relaxed);
  return SRES_OK;
}

extern "C" int sres_l2_persist_window(const void* base, size_t bytes, void* stream) {
  cudaStreamAttrValue v;
  memset(&v, 0, sizeof(v));
  if (base && bytes) {
    int dev = 0, max_win = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&max_win, cudaDevAttrMaxAccessPolicyWindowSize, dev);
    if (max_win > 0 && bytes > (size_t)max_win) bytes = (size_t)max_win;
    v.accessPolicyWindow.base_ptr = const_cast<void*>(base);
    v.accessPolicyWindow.num_bytes = bytes;
    v.accessPolicyWindow.hitRatio = 1.0f;
    v.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
    v.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
  } else {
    v.accessPolicyWindow.num_bytes = 0;
    v.accessPolicyWindow.hitProp = cudaAccessPropertyNormal;
    v.accessPolicyWindow.missProp = cudaAccessPropertyNormal;
  }
  cudaError_t e = cudaStreamSetAttribute((cudaStream_t)stream, cudaStreamAttributeAccessPolicyWindow, &v);
  if (e != cudaSuccess) return sres::set_cuda_error(e, "l2_persist_window: cudaStreamSetAttribute");
  return SRES_OK;
}
