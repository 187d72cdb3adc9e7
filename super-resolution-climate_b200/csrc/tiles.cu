// Tile extraction / normalisation / stitching on the device -- pure data movement (HBM-bound,
// index-exact) around the model.
//
//   tiles_finite_flags  which candidate tiles survive the reference's NaN-tile drop
//                       (sres/base/source/swot/raw.py:226: isfinite(tile.mean(-1).mean(-1)))
//   tiles_gather        region (C,Y,X) -> tiles (N,C,Th,Tw) through an explicit source-tile table, so
//                       both the reference's channel-major order and the corrected tile-major order
//                       are the same kernel (raw.py:216-233)
//   tiles_lnorm         per tile, per channel (x-mean)/std, NaN-skipping, population std, with the
//                       8-way xyflip fused into the store (raw.py:176-183; source/batch.py:37-49)
//   tiles_stitch        tiles -> (gy*th, gx*tw) image, NaN where no tile landed, optional de-normalise
//                       x*std+mean (dual_trainer.py:449-480, :67-77)
#include <math.h>
#include "internal.h"

namespace sres {

__global__ void __launch_bounds__(256)
tiles_finite_flags_kernel(const float* __restrict__ region, int C, int Y, int X, int y0, int x0, int Th, int Tw, int gy,
                          int gx, int* __restrict__ flags) {
  const int cand = blockIdx.x;  // c*gy*gx + ty*gx + tx
  const int tx = cand % gx, ty = (cand / gx) % gy, c = cand / (gx * gy);
  const float* base = region + ((size_t)c * Y + (y0 + (size_t)ty * Th)) * X + x0 + (size_t)tx * Tw;
  int ok = 1;
  for (int i = threadIdx.x; i < Th * Tw; i += blockDim.x) {
    const float v = base[(size_t)(i / Tw) * X + (i % Tw)];
    if (!isfinite(v)) ok = 0;
  }
  ok = __syncthreads_and(ok);
  if (threadIdx.x == 0) flags[cand] = ok;
}

__global__ void __launch_bounds__(256)
tiles_gather_kernel(const float* __restrict__ region, int C, int Y, int X, int y0, int x0, int Th, int Tw, int gy, int gx,
                    const int* __restrict__ src, float* __restrict__ out) {
  const int slot = blockIdx.x;  // n*C + c of the output
  const int cand = src[slot];
  const int tx = cand % gx, ty = (cand / gx) % gy, c = cand / (gx * gy);
  const float* base = region + ((size_t)c * Y + (y0 + (size_t)ty * Th)) * X + x0 + (size_t)tx * Tw;
  float* o = out + (size_t)slot * Th * Tw;
  for (int i = threadIdx.x; i < Th * Tw; i += blockDim.x) o[i] = base[(size_t)(i / Tw) * X + (i % Tw)];
}

__global__ void __launch_bounds__(256)
tiles_lnorm_kernel(const float* __restrict__ in, int Th, int Tw, int flip, float* __restrict__ out,
                   float* __restrict__ mean_out, float* __restrict__ std_out) {
  __shared__ double sm[256];
  __shared__ int sc[256];
  __shared__ float s_mean, s_std;
  const int n = Th * Tw;
  const float* ip = in + (size_t)blockIdx.x * n;
  float* op = out + (size_t)blockIdx.x * n;
  double a = 0.0;
  int cnt = 0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float v = ip[i];
    if (!isnan(v)) { a += (double)v; ++cnt; }
  }
  sm[threadIdx.x] = a; sc[threadIdx.x] = cnt;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (threadIdx.x < s) { sm[threadIdx.x] += sm[threadIdx.x + s]; sc[threadIdx.x] += sc[threadIdx.x + s]; }
    __syncthreads();
  }
  const int total = sc[0];
  const double mean = sm[0] / (double)total;
  __syncthreads();
  a = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float v = ip[i];
    if (!isnan(v)) { const double d = (double)v - mean; a += d * d; }
  }
  sm[threadIdx.x] = a;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (threadIdx.x < s) sm[threadIdx.x] += sm[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    s_mean = (float)mean;
    s_std = (float)sqrt(sm[0] / (double)total);
    mean_out[blockIdx.x] = s_mean;
    std_out[blockIdx.x] = s_std;
  }
  __syncthreads();
  const float m = s_mean, sd = s_std;
  // the flipped plane is Th x Tw for flips 0-3 and Tw x Th for flips 4-7 (the transpose comes last)
  const int ow = (flip & 4) ? Th : Tw;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    // out[y][x] of the flipped batch <- in[sy][sx]  (flip x, then flip y, then transpose)
    int y = i / ow, x = i % ow;
    if (flip & 4) { const int t = y; y = x; x = t; }
    if (flip & 2) y = Th - 1 - y;
    if (flip & 1) x = Tw - 1 - x;
    op[i] = __fdiv_rn(__fsub_rn(ip[y * Tw + x], m), sd);
  }
}

__global__ void __launch_bounds__(256)
tiles_stitch_kernel(const float* __restrict__ tiles, int C, int ivar, int th, int tw, int gy, int gx,
                    const int* __restrict__ cell_to_tile, const float* __restrict__ mean, const float* __restrict__ std_,
                    float* __restrict__ out) {
  const long long total = (long long)gy * th * gx * tw;
  const int Wimg = gx * tw;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int X = int(i % Wimg), Yp = int(i / Wimg);
    const int cell = (Yp / th) * gx + (X / tw);
    const int n = cell_to_tile[cell];
    float v = nanf("");
    if (n >= 0) {
      v = tiles[(((size_t)n * C + ivar) * th + (Yp % th)) * tw + (X % tw)];
      if (mean) v = __fadd_rn(__fmul_rn(v, std_[n * C + ivar]), mean[n * C + ivar]);
    }
    out[i] = v;
  }
}

}  // namespace sres

using namespace sres;

static int tiles_geom_ok(int C, int Y, int X, int y0, int x0, int Th, int Tw, int gy, int gx) {
  if (C <= 0 || Th <= 0 || Tw <= 0 || gy <= 0 || gx <= 0 || y0 < 0 || x0 < 0) return 0;
  if ((long long)y0 + (long long)gy * Th > Y || (long long)x0 + (long long)gx * Tw > X) return 0;
  return 1;
}

extern "C" int sres_tiles_finite_flags_hw(const float* region, int C, int Y, int X, int y0, int x0, int Th, int Tw, int gy,
                                          int gx, int32_t* flags, void* stream) {
  if (!region || !flags) return set_error(SRES_ERR_INVALID_ARG, "tiles_finite_flags: null pointer");
  if (!tiles_geom_ok(C, Y, X, y0, x0, Th, Tw, gy, gx)) return set_error(SRES_ERR_INVALID_ARG, "tiles: grid exceeds region");
  tiles_finite_flags_kernel<<<C * gy * gx, 256, 0, (cudaStream_t)stream>>>(region, C, Y, X, y0, x0, Th, Tw, gy, gx, flags);
  SRES_CHECK_LAUNCH("tiles_finite_flags: launch");
  return SRES_OK;
}

extern "C" int sres_tiles_gather_hw(const float* region, int C, int Y, int X, int y0, int x0, int Th, int Tw, int gy, int gx,
                                    const int32_t* src_tile, int nslots, float* out, void* stream) {
  if (!region || !src_tile || !out) return set_error(SRES_ERR_INVALID_ARG, "tiles_gather: null pointer");
  if (!tiles_geom_ok(C, Y, X, y0, x0, Th, Tw, gy, gx)) return set_error(SRES_ERR_INVALID_ARG, "tiles: grid exceeds region");
  if (nslots <= 0) return SRES_OK;
  tiles_gather_kernel<<<nslots, 256, 0, (cudaStream_t)stream>>>(region, C, Y, X, y0, x0, Th, Tw, gy, gx, src_tile, out);
  SRES_CHECK_LAUNCH("tiles_gather: launch");
  return SRES_OK;
}

extern "C" int sres_tiles_lnorm_hw(const float* in, int nplanes, int Th, int Tw, int flip_index, float* out, float* mean,
                                   float* std_, void* stream) {
  if (!in || !out || !mean || !std_) return set_error(SRES_ERR_INVALID_ARG, "tiles_lnorm: null pointer");
  if (nplanes <= 0 || Th <= 0 || Tw <= 0 || flip_index < 0 || flip_index > 7)
    return set_error(SRES_ERR_INVALID_ARG, "tiles_lnorm: bad argument");
  if (in == out && flip_index != 0) return set_error(SRES_ERR_INVALID_ARG, "tiles_lnorm: in-place needs flip_index 0");
  tiles_lnorm_kernel<<<nplanes, 256, 0, (cudaStream_t)stream>>>(in, Th, Tw, flip_index, out, mean, std_);
  SRES_CHECK_LAUNCH("tiles_lnorm: launch");
  return SRES_OK;
}

extern "C" int sres_tiles_stitch_hw(const float* tiles, int C, int ivar, int th, int tw, int gy, int gx,
                                    const int32_t* cell_to_tile, const float* mean, const float* std_, float* out,
                                    void* stream) {
  if (!tiles || !cell_to_tile || !out) return set_error(SRES_ERR_INVALID_ARG, "tiles_stitch: null pointer");
  if (C <= 0 || ivar < 0 || ivar >= C || th <= 0 || tw <= 0 || gy <= 0 || gx <= 0 || (mean == nullptr) != (std_ == nullptr))
    return set_error(SRES_ERR_INVALID_ARG, "tiles_stitch: bad argument");
  const long long total = (long long)gy * th * gx * tw;
  int sms = device_sm_count();
  if (sms <= 0) sms = 148;
  long long blocks = (total + 255) / 256;
  if (blocks > sms * 16LL) blocks = sms * 16LL;
  tiles_stitch_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(tiles, C, ivar, th, tw, gy, gx, cell_to_tile, mean,
                                                                       std_, out);
  SRES_CHECK_LAUNCH("tiles_stitch: launch");
  return SRES_OK;
}

// square tiles: the original entry points, T = Th = Tw
extern "C" int sres_tiles_finite_flags(const float* region, int C, int Y, int X, int y0, int x0, int T, int gy, int gx,
                                       int32_t* flags, void* stream) {
  return sres_tiles_finite_flags_hw(region, C, Y, X, y0, x0, T, T, gy, gx, flags, stream);
}

extern "C" int sres_tiles_gather(const float* region, int C, int Y, int X, int y0, int x0, int T, int gy, int gx,
                                 const int32_t* src_tile, int nslots, float* out, void* stream) {
  return sres_tiles_gather_hw(region, C, Y, X, y0, x0, T, T, gy, gx, src_tile, nslots, out, stream);
}

extern "C" int sres_tiles_lnorm(const float* in, int nplanes, int T, int flip_index, float* out, float* mean,
                                float* std_, void* stream) {
  return sres_tiles_lnorm_hw(in, nplanes, T, T, flip_index, out, mean, std_, stream);
}

extern "C" int sres_tiles_stitch(const float* tiles, int C, int ivar, int t, int gy, int gx, const int32_t* cell_to_tile,
                                 const float* mean, const float* std_, float* out, void* stream) {
  return sres_tiles_stitch_hw(tiles, C, ivar, t, t, gy, gx, cell_to_tile, mean, std_, out, stream);
}
