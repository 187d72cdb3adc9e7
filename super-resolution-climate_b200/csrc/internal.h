// Host-side helpers shared by the translation units of libsres_b200.so.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/sres_b200.h"

namespace sres {

// thread-local last-error text + status passthrough
int set_error(int code, const char* msg);
int set_cuda_error(cudaError_t e, const char* where);

// cached SM count of the current device (<=0 when there is none)
int device_sm_count();
// grid of a persistent kernel that walks n_tiles equal tiles: one CTA per SM, or per tile when there are fewer
int persistent_grid(int n_tiles, int sms);

// 2-D TMA descriptor over a row-major [nrows][64] bf16 matrix (128-byte rows), box = 64 x box_rows,
// 128B swizzle, zero fill outside [0, nrows).
int make_tmap_rows64(CUtensorMap* out, const void* base, uint64_t nrows, uint32_t box_rows);

// 2-D TMA descriptor over a row-major [nrows][64] fp32 matrix (256-byte rows), box = 32 floats x box_rows
// (one 128B-swizzled half row), zero fill outside [0, nrows).
int make_tmap_rows64_f32(CUtensorMap* out, const void* base, uint64_t nrows, uint32_t box_rows);

// 2-D TMA descriptor over a [nrows][64] bf16 matrix with a HALF-row box (32 channels = 64 bytes) x box_rows,
// 64B swizzle: the per-warp epilogue slabs of the conv kernel.
int make_tmap_rows64_half(CUtensorMap* out, const void* base, uint64_t nrows, uint32_t box_rows);

// Launch with the programmatic-stream-serialization attribute (PDL).  SRES_PDL=0 in the environment turns
// the attribute off (plain stream order) for A/B measurements.
bool l2_hint_enabled();  // true after sres_l2_set_aside(bytes > 0)
bool pdl_enabled();
int pdl_level();  // SRES_PDL: 0 = off, 1 = tensor-core kernels only, 2 = also the channel-attention kernels (default)
// Process-wide count of kernels this library has enqueued (eagerly or into a stream capture): sres_launch_count().  The host
// engine reads it around its forward / backward calls so that bench.py's `gpu_launches` is counted, not derived.
void count_launch();
template <typename... KArgs, typename... Args>
cudaError_t launch_pdl_if(bool on, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = on ? 1 : 0;
  count_launch();
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  count_launch();
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// three-taps-per-MMA tail convolution (conv_n192.cu, N = 48): 64 -> c_real <= 16 with planar fp32 output, any image width
bool conv_n48_available(int H, int W);
int launch_conv_n48(const sres_conv_args* a, cudaStream_t stream);

#define SRES_CHECK_LAUNCH(where)                                  \
  do {                                                            \
    cudaError_t e__ = cudaGetLastError();                         \
    if (e__ != cudaSuccess) return sres::set_cuda_error(e__, where); \
    sres::count_launch();                                         \
  } while (0)

}  // namespace sres
