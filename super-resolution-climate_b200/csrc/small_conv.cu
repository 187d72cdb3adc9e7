// The narrow 3x3 convolutions at the two ends of RCAN, on CUDA cores (they are HBM-bound: K or N
// is only 9*C with C = 1..16 image channels, SURVEY.md section 2 op inventory).
//
//   conv3x3_small_in   : planar fp32 NCHW (C_s channels) -> 64-feature PTL rows.
//                        head conv forward (sres/model/rcan/network.py:13,23) and, with transposed +
//                        flipped weights, the input-gradient of the tail conv (network.py:16).
//   small_in_wgrad     : weight/bias gradient of the head conv (reduction over all positions).
//   small_out_wgrad    : weight/bias gradient of the tail conv 64 -> C_s.
//
// The kernels are written for at most kChunkC = 4 channels.  More channels (up to kMaxSmallC = 16):
//   * the weight gradients and the CUDA-core tail forward compute every output element from one image channel, so they
//     run as ceil(C_s / 4) launches over channel chunks (Ctot = the image's channel count, c0 = the chunk's first);
//   * the head forward and the tail input-gradient sum over the channels: conv3x3_small_in_wide_kernel (weights in
//     shared memory, narrower column strips) takes 5..16 channels in one launch.
#include "internal.h"
#include "ptx.cuh"

namespace sres {

constexpr int kChunkC = 4;
constexpr int kMaxSmallC = 16;

// ---------------------------------------------------------------------------------------------
// planar (B,Cs,H,W) fp32  ->  PTL [rows][64]
//   transposed == 0:  w is (64, Cs, 3, 3):  out[q][n] = b[n] + sum_{c,t} w[n][c][t] * in[c][q+off(t)]
//   transposed == 1:  w is (Cs, 64, 3, 3):  out[q][n] =        sum_{c,t} w[c][n][8-t] * in[c][q+off(t)]
// A block owns a band of kBandRows image rows of one image: the planar input band (+1 row/column halo,
// zero outside the image) is staged in shared memory once; a thread owns 2 output features (its 2*Cs*9
// weights live in registers) and walks the band's PTL rows, so a warp writes one full 128-byte bf16 row
// (256-byte fp32 row) per position.  Padding rows (x == W, y == H) are written as zeros.
// ---------------------------------------------------------------------------------------------
constexpr int kBandRows = 8;

// Wide images are walked in column strips of at most 256 pixels (a multiple of 4), so the staged band stays below 48 KB
// and two blocks share an SM: with the whole 768-pixel row of the x8 configuration staged (123 KB) one block of 8 warps
// per SM left the issue slots 48 % busy (ncu, round 2) -- the kernels are instruction-bound, not HBM-bound.
__host__ __device__ inline int strip_cols(int W) {
  const int n = (W + 255) / 256;
  return (((W + n - 1) / n) + 3) & ~3;
}

// Stage the planar fp32 band rows [y0-1, y0+kBandRows] x columns [x_lo-1, x_lo+S] of channels c0 .. c0+nch-1 of image b
// (Ctot channels an image; zero outside the image) as s[c - c0][r][i], i = column - (x_lo - 1), pitch SWp.  One warp per
// (channel, row): coalesced, no per-element division.
// Asynchronous copies (cp.async, zero-fill outside the image): the callers stage item i+1 into the other half of a double
// buffer while they compute item i -- staged synchronously, the ~40 dependent global loads per thread and item took as
// long as the item's arithmetic.
__device__ __forceinline__ void stage_band_async(float* s, const float* __restrict__ in, int nch, int Ctot, int c0, int b,
                                                 int H, int W, int y0, int x_lo, int SWp) {
  const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
  for (int cr = wrp; cr < nch * (kBandRows + 2); cr += 8) {
    const int c = cr / (kBandRows + 2), r = cr - c * (kBandRows + 2), yy = y0 - 1 + r;
    const bool yin = yy >= 0 && yy < H;
    const float* src = in + (((size_t)b * Ctot + c0 + c) * H + (yin ? yy : 0)) * W;
    float* dst = s + cr * SWp;
    for (int i = lane; i < SWp; i += 32) {
      const int xx = x_lo - 1 + i;
      const bool ok = yin && xx >= 0 && xx < W;
      cp_async4_zfill(dst + i, src + (ok ? xx : 0), ok ? 4 : 0);
    }
  }
}

// item -> (image, first band row, first strip column)
struct BandItem { int b, y0, x_lo; };
__device__ __forceinline__ BandItem band_item(int item, int bands, int nstrips, int S) {
  const int strip = item % nstrips, bb = item / nstrips;
  return BandItem{bb / bands, (bb % bands) * kBandRows, strip * S};
}

template <int CS>
__global__ void __launch_bounds__(256, 2)
conv3x3_small_in_kernel(const float* __restrict__ in, const float* __restrict__ w, const float* __restrict__ bias,
                        int B, int H, int W, int transposed, int unshuffle, float* __restrict__ out_f32,
                        uint16_t* __restrict__ out_bf16) {
  extern __shared__ float s_buf[];  // 2 x [CS][kBandRows+2][S+2]
  const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
  const int n0 = lane * 2;  // two output features
  float2 wr[CS * 9], br;   // .x / .y = the thread's two features: packed FMAs (ffma2_bcast)
  {
    float wt[2][CS * 9], bt[2];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      bt[j] = (bias && !transposed) ? bias[n0 + j] : 0.f;
#pragma unroll
      for (int c = 0; c < CS; ++c)
#pragma unroll
        for (int t = 0; t < 9; ++t)
          wt[j][c * 9 + t] = transposed ? w[(c * 64 + n0 + j) * 9 + (8 - t)] : w[((n0 + j) * CS + c) * 9 + t];
    }
    br = make_float2(bt[0], bt[1]);
#pragma unroll
    for (int i = 0; i < CS * 9; ++i) wr[i] = make_float2(wt[0][i], wt[1][i]);
  }
  const int P = W + 1, RP = (H + 1) * P;
  const int S = strip_cols(W), nstrips = (W + S - 1) / S, SWp = S + 2;   // even pitch: 8-byte aligned pairs
  const int bands = (H + 1 + kBandRows - 1) / kBandRows;  // the zero row y == H belongs to the last band
  const int f = unshuffle > 1 ? unshuffle : 1;
  const int Pl = W / f + 1, Rl = H / f + 1;
  // PTL row of pixel (y, x) of image b: plain, or PixelUnshuffle(f): sub-grid (y%f, x%f), position (y/f, x/f)
  auto row_of = [&](int b, int y, int subx) -> long long {
    if (f == 1) return (long long)b * RP + (long long)y * P;
    return ((long long)((y % f) * f + subx) * B + b) * Rl * Pl + (long long)(y / f) * Pl;
  };
  auto put = [&](long long oq, float a0, float a1) {
    if (out_f32) *reinterpret_cast<float2*>(out_f32 + oq * 64 + n0) = make_float2(a0, a1);
    if (out_bf16) *reinterpret_cast<uint32_t*>(out_bf16 + oq * 64 + n0) = pack_bf16x2(a0, a1);
  };
  auto store = [&](int b, int y, int x, float a0, float a1) { put(row_of(b, y, x % f) + x / f, a0, a1); };
  const int n_items = B * bands * nstrips, buf_floats = CS * (kBandRows + 2) * SWp;
  if ((int)blockIdx.x < n_items) {
    const BandItem it = band_item(blockIdx.x, bands, nstrips, S);
    stage_band_async(s_buf, in, CS, CS, 0, it.b, H, W, it.y0, it.x_lo, SWp);
  }
  cp_async_commit();
  int parity = 0;
  for (int item = blockIdx.x; item < n_items; item += gridDim.x, parity ^= 1) {
    const BandItem it = band_item(item, bands, nstrips, S);
    const int b = it.b, y0 = it.y0, x_lo = it.x_lo, x_hi = min(W, x_lo + S);
    const bool last_strip = x_lo + S >= W;
    const float* s_in = s_buf + parity * buf_floats;
    __syncthreads();   // every warp is done with the previous item: its buffer is free for the prefetch
    if (item + (int)gridDim.x < n_items) {
      const BandItem nx = band_item(item + gridDim.x, bands, nstrips, S);
      stage_band_async(s_buf + (parity ^ 1) * buf_floats, in, CS, CS, 0, nx.b, H, W, nx.y0, nx.x_lo, SWp);
    }
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();
    const int rows = min(kBandRows, H + 1 - y0);
    if ((W & 3) == 0) {
      // four consecutive positions per step (plus one step per row for the padding column): the 6 inputs a 3-tap row
      // needs come from three aligned 8-byte shared loads, 18 loads feed 144 FMAs instead of 72 scalar loads
      // Rows outside, groups inside, row pointers hoisted: the integer work per step (a division by the groups per row,
      // 64-bit PTL row arithmetic for every store) ran on the same pipe as the FMAs and was 15 % of the instructions.
      const int ng = (x_hi - x_lo) >> 2;
      for (int yl = 0; yl < rows; ++yl) {
        const int y = y0 + yl;
        if (y == H || (f != 1 && f != 2)) {
          // the zero row below the image / an unusual unshuffle factor: position by position
          const int ncol = x_hi - x_lo + (last_strip ? 1 : 0);
          for (int xr = wrp; xr < ncol; xr += 8) {
            const int x = x_lo + xr;
            float2 a = make_float2(0.f, 0.f);
            if (x != W && y != H) {
              a = br;
#pragma unroll
              for (int c = 0; c < CS; ++c)
#pragma unroll
                for (int t = 0; t < 9; ++t)
                  ffma2_bcast(a, wr[c * 9 + t], s_in[(c * (kBandRows + 2) + yl + t / 3) * SWp + xr + t % 3]);
            }
            store(b, y, x, a.x, a.y);
          }
          continue;
        }
        // f == 1: positions x0..x0+3 are rows q0 + x0 + j;  f == 2: rows q0 + x0/2 (+1) of sub-grid 0 and q1 + ... of sub-grid 1
        const long long q0 = row_of(b, y, 0), q1 = f == 2 ? row_of(b, y, 1) : q0;
        float* const f0 = out_f32 ? out_f32 + q0 * 64 + n0 : nullptr;
        float* const f1 = out_f32 ? out_f32 + q1 * 64 + n0 : nullptr;
        uint16_t* const h0 = out_bf16 ? out_bf16 + q0 * 64 + n0 : nullptr;
        uint16_t* const h1 = out_bf16 ? out_bf16 + q1 * 64 + n0 : nullptr;
        const float* srow = s_in + yl * SWp;
        for (int gi = wrp; gi < ng; gi += 8) {
          const int xr = gi * 4;
          float2 a[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) a[j] = br;
#pragma unroll
          for (int c = 0; c < CS; ++c)
#pragma unroll
            for (int ty = 0; ty < 3; ++ty) {
              const float* dr = srow + (c * (kBandRows + 2) + ty) * SWp + xr;
              const float2 d01 = *reinterpret_cast<const float2*>(dr);
              const float2 d23 = *reinterpret_cast<const float2*>(dr + 2);
              const float2 d45 = *reinterpret_cast<const float2*>(dr + 4);
              const float d6[6] = {d01.x, d01.y, d23.x, d23.y, d45.x, d45.y};
#pragma unroll
              for (int tx = 0; tx < 3; ++tx)
#pragma unroll
                for (int j = 0; j < 4; ++j) ffma2_bcast(a[j], wr[c * 9 + ty * 3 + tx], d6[j + tx]);
            }
          // element offsets of the four positions from the row pointers (32-bit: a row of the image is < 2^31 elements)
          const int e0 = f == 2 ? ((x_lo + xr) >> 1) * 64 : (x_lo + xr) * 64;
          const int step = f == 2 ? 0 : 64;   // f == 2: positions 0/1 share a row of their sub-grids, 2/3 the next one
          const int e[4] = {e0, e0 + step, e0 + 64 + step, e0 + 64 + 2 * step};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const bool odd = f == 2 && (j & 1);
            if (out_f32) *reinterpret_cast<float2*>((odd ? f1 : f0) + e[j]) = a[j];
            if (out_bf16) *reinterpret_cast<uint32_t*>((odd ? h1 : h0) + e[j]) = pack_bf16x2(a[j].x, a[j].y);
          }
        }
        if (last_strip && wrp == (ng & 7)) store(b, y, W, 0.f, 0.f);   // the padding column
      }
      continue;
    }
    const int ncol = x_hi - x_lo + (last_strip ? 1 : 0);   // + the padding column x == W
    for (int pos = wrp; pos < rows * ncol; pos += 8) {
      const int yl = pos / ncol, xr = pos - yl * ncol, x = x_lo + xr, y = y0 + yl;
      float2 a = make_float2(0.f, 0.f);
      if (x != W && y != H) {
        a = br;
#pragma unroll
        for (int c = 0; c < CS; ++c)
#pragma unroll
          for (int t = 0; t < 9; ++t)
            ffma2_bcast(a, wr[c * 9 + t], s_in[(c * (kBandRows + 2) + yl + t / 3) * SWp + xr + t % 3]);
      }
      store(b, y, x, a.x, a.y);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// conv3x3_small_in for 5..16 channels (same math, same PTL row mappings, same padding rows).  The kernel above cannot
// simply be instantiated with CS = 16: its 2*CS*9 weights a thread would be 288 registers, and its double-buffered
// 256-column band 333 KB.  Here
//   * the weights sit in shared memory as feature pairs, float2 sw[c*9 + t][32] (lane l holds features 2l, 2l+1): a
//     warp reads one 256-byte row per tap and channel, shared by four positions;
//   * the column strips are at most kWideStrip pixels: at 16 channels the two band buffers and the weights take 98.5 KB,
//     so two blocks share an SM;
//   * a warp walks groups of four consecutive positions of the whole band (W % 4 == 0), any unshuffle factor, or single
//     positions otherwise; the channel loop is not unrolled (its body is 36 FFMA2 for 18 shared loads).
// Accumulation is fp32, channel by channel and tap by tap, as above.
// ---------------------------------------------------------------------------------------------
constexpr int kWideStrip = 48;

__host__ __device__ inline int strip_cols_wide(int W) {
  const int n = (W + kWideStrip - 1) / kWideStrip;
  return (((W + n - 1) / n) + 3) & ~3;
}

__host__ __device__ inline size_t small_in_wide_smem_bytes(int Cs, int W) {
  return (2 * (size_t)Cs * (kBandRows + 2) * (strip_cols_wide(W) + 2) + (size_t)Cs * 9 * 64) * sizeof(float);
}

__global__ void __launch_bounds__(256, 2)
conv3x3_small_in_wide_kernel(const float* __restrict__ in, const float* __restrict__ w, const float* __restrict__ bias,
                             int B, int Cs, int H, int W, int transposed, int unshuffle, float* __restrict__ out_f32,
                             uint16_t* __restrict__ out_bf16) {
  extern __shared__ float s_buf[];  // 2 x [Cs][kBandRows+2][S+2], then the weights [Cs*9][64]
  const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
  const int n0 = lane * 2;
  const int S = strip_cols_wide(W), nstrips = (W + S - 1) / S, SWp = S + 2;   // even pitch: 8-byte aligned pairs
  const int buf_floats = Cs * (kBandRows + 2) * SWp;
  float* const s_w = s_buf + 2 * buf_floats;
  for (int i = threadIdx.x; i < Cs * 9 * 64; i += blockDim.x) {
    const int n = i & 63, ct = i >> 6, c = ct / 9, t = ct - c * 9;
    s_w[i] = transposed ? w[(c * 64 + n) * 9 + (8 - t)] : w[(n * Cs + c) * 9 + t];
  }
  const float2* const sw2 = reinterpret_cast<const float2*>(s_w) + lane;
  const float2 br = (bias && !transposed) ? make_float2(bias[n0], bias[n0 + 1]) : make_float2(0.f, 0.f);
  const int P = W + 1, RP = (H + 1) * P;
  const int bands = (H + 1 + kBandRows - 1) / kBandRows;  // the zero row y == H belongs to the last band
  const int f = unshuffle > 1 ? unshuffle : 1;
  const int Pl = W / f + 1, Rl = H / f + 1;
  auto row_of = [&](int b, int y, int subx) -> long long {
    if (f == 1) return (long long)b * RP + (long long)y * P;
    return ((long long)((y % f) * f + subx) * B + b) * Rl * Pl + (long long)(y / f) * Pl;
  };
  auto store = [&](int b, int y, int x, float a0, float a1) {
    const long long oq = row_of(b, y, x % f) + x / f;
    if (out_f32) *reinterpret_cast<float2*>(out_f32 + oq * 64 + n0) = make_float2(a0, a1);
    if (out_bf16) *reinterpret_cast<uint32_t*>(out_bf16 + oq * 64 + n0) = pack_bf16x2(a0, a1);
  };
  const int n_items = B * bands * nstrips;
  if ((int)blockIdx.x < n_items) {
    const BandItem it = band_item(blockIdx.x, bands, nstrips, S);
    stage_band_async(s_buf, in, Cs, Cs, 0, it.b, H, W, it.y0, it.x_lo, SWp);
  }
  cp_async_commit();
  int parity = 0;
  for (int item = blockIdx.x; item < n_items; item += gridDim.x, parity ^= 1) {
    const BandItem it = band_item(item, bands, nstrips, S);
    const int b = it.b, y0 = it.y0, x_lo = it.x_lo, x_hi = min(W, x_lo + S);
    const bool last_strip = x_lo + S >= W;
    const float* s_in = s_buf + parity * buf_floats;
    __syncthreads();   // every warp is done with the previous item (and the weights are in place, first time round)
    if (item + (int)gridDim.x < n_items) {
      const BandItem nx = band_item(item + gridDim.x, bands, nstrips, S);
      stage_band_async(s_buf + (parity ^ 1) * buf_floats, in, Cs, Cs, 0, nx.b, H, W, nx.y0, nx.x_lo, SWp);
    }
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();
    const int rows = min(kBandRows, H + 1 - y0);
    const int img_rows = min(kBandRows, H - y0);   // rows above the zero row y == H
    const int ncol = x_hi - x_lo + (last_strip ? 1 : 0);   // + the padding column x == W
    if ((W & 3) == 0) {
      const int ng = (x_hi - x_lo) >> 2;
      for (int g = wrp; g < img_rows * ng; g += 8) {
        const int yl = g / ng, xr = (g - yl * ng) * 4;
        float2 a[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) a[j] = br;
#pragma unroll 1
        for (int c = 0; c < Cs; ++c) {
          const float* srow = s_in + (c * (kBandRows + 2) + yl) * SWp + xr;
          const float2* wc = sw2 + c * 9 * 32;
#pragma unroll
          for (int ty = 0; ty < 3; ++ty) {
            const float* dr = srow + ty * SWp;
            const float2 d01 = *reinterpret_cast<const float2*>(dr);
            const float2 d23 = *reinterpret_cast<const float2*>(dr + 2);
            const float2 d45 = *reinterpret_cast<const float2*>(dr + 4);
            const float d6[6] = {d01.x, d01.y, d23.x, d23.y, d45.x, d45.y};
#pragma unroll
            for (int tx = 0; tx < 3; ++tx) {
              const float2 wv = wc[(ty * 3 + tx) * 32];
#pragma unroll
              for (int j = 0; j < 4; ++j) ffma2_bcast(a[j], wv, d6[j + tx]);
            }
          }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) store(b, y0 + yl, x_lo + xr + j, a[j].x, a[j].y);
      }
      // zeros: the padding column of the image rows, then the zero row y == H if it is in this band
      if (last_strip)
        for (int yl = wrp; yl < img_rows; yl += 8) store(b, y0 + yl, W, 0.f, 0.f);
      if (rows > img_rows)
        for (int xr = wrp; xr < ncol; xr += 8) store(b, H, x_lo + xr, 0.f, 0.f);
      continue;
    }
    for (int pos = wrp; pos < rows * ncol; pos += 8) {
      const int yl = pos / ncol, xr = pos - yl * ncol, x = x_lo + xr, y = y0 + yl;
      float2 a = make_float2(0.f, 0.f);
      if (x != W && y != H) {
        a = br;
#pragma unroll 1
        for (int c = 0; c < Cs; ++c)
#pragma unroll
          for (int t = 0; t < 9; ++t)
            ffma2_bcast(a, sw2[(c * 9 + t) * 32], s_in[(c * (kBandRows + 2) + yl + t / 3) * SWp + xr + t % 3]);
      }
      store(b, y, x, a.x, a.y);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// head-conv weight gradient: dW[n][c][t] = sum_q (g1+g2)[q][n] * in[c][q+off(t)],  db[n] = sum_q g[q][n]
// block = 64 features x 4 position lanes; per-block partials then a fixed-order reduce.
// One launch covers Cs <= kChunkC channels c0 .. c0+Cs-1 of an image with Ctot channels.
// ---------------------------------------------------------------------------------------------
constexpr int kSwAcc = kChunkC * 9 + 1;

__global__ void __launch_bounds__(256)
small_in_wgrad_kernel(const float* __restrict__ g1, const float* __restrict__ g2, const float* __restrict__ in, int B,
                      int Cs, int Ctot, int c0, int H, int W, float* __restrict__ part) {
  __shared__ float sm[4][64][kSwAcc];
  const int n = threadIdx.x & 63, ln = threadIdx.x >> 6;
  const int P = W + 1, RP = (H + 1) * P;
  const long long npos = (long long)B * RP;
  float acc[kSwAcc];
#pragma unroll
  for (int i = 0; i < kSwAcc; ++i) acc[i] = 0.f;
  for (long long q = (long long)blockIdx.x * 4 + ln; q < npos; q += (long long)gridDim.x * 4) {
    const int b = int(q / RP), rem = int(q - (long long)b * RP);
    const int y = rem / P, x = rem - y * P;
    if (x == W || y == H) continue;
    float gv = g1[q * 64 + n];
    if (g2) gv += g2[q * 64 + n];
    acc[kSwAcc - 1] += gv;
    for (int c = 0; c < Cs; ++c) {
      const float* ip = in + ((size_t)b * Ctot + c0 + c) * H * W;
#pragma unroll
      for (int t = 0; t < 9; ++t) {
        const int yy = y + t / 3 - 1, xx = x + t % 3 - 1;
        if (yy < 0 || yy >= H || xx < 0 || xx >= W) continue;
        acc[c * 9 + t] = fmaf(gv, __ldg(ip + (size_t)yy * W + xx), acc[c * 9 + t]);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < kSwAcc; ++i) sm[ln][n][i] = acc[i];
  __syncthreads();
  for (int i = threadIdx.x; i < 64 * kSwAcc; i += 256) {
    const int nn = i / kSwAcc, e = i % kSwAcc;
    part[(size_t)blockIdx.x * 64 * kSwAcc + i] = sm[0][nn][e] + sm[1][nn][e] + sm[2][nn][e] + sm[3][nn][e];
  }
}

// Band-tiled head-conv weight gradient for W % 4 == 0 (the mirror image of small_out_wgrad_kernel below): the planar
// input band (+halo) sits in shared memory, a thread owns 2 features of the fp32 gradient rows (g1 + g2), a warp walks
// groups of four consecutive positions and reads the 6 inputs of a 3-tap row with three 8-byte shared loads.  The
// scalar kernel above keeps its loads under boundary branches and was latency-bound (208 us for 78 MB).
template <int CS>
__global__ void __launch_bounds__(256)
small_in_wgrad_band_kernel(const float* __restrict__ g1, const float* __restrict__ g2, const float* __restrict__ in, int B,
                           int Ctot, int c0, int H, int W, float* __restrict__ part) {
  extern __shared__ float s_x[];  // [CS][kBandRows+2][SW], then the cross-warp reduction buffer
  const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
  const int n0 = lane * 2;
  const int P = W + 1, RP = (H + 1) * P, SW = (W + 3) & ~1;
  float acc[2][CS * 9], accb[2] = {0.f, 0.f};
#pragma unroll
  for (int j = 0; j < 2; ++j)
#pragma unroll
    for (int i = 0; i < CS * 9; ++i) acc[j][i] = 0.f;
  const int bands = (H + kBandRows - 1) / kBandRows;
  const int gpr = W >> 2;
  for (int item = blockIdx.x; item < B * bands; item += gridDim.x) {
    const int b = item / bands, y0 = (item % bands) * kBandRows;
    __syncthreads();
    for (int i = threadIdx.x; i < CS * (kBandRows + 2) * SW; i += blockDim.x) {
      const int xx = i % SW - 1, yy = (i / SW) % (kBandRows + 2) + y0 - 1, c = i / (SW * (kBandRows + 2));
      s_x[i] = (yy >= 0 && yy < H && xx >= 0 && xx < W) ? __ldg(in + (((size_t)b * Ctot + c0 + c) * H + yy) * W + xx) : 0.f;
    }
    __syncthreads();
    const int rows = min(kBandRows, H - y0);
    for (int grp = wrp; grp < rows * gpr; grp += 8) {
      const int yl = grp / gpr, x0 = (grp - yl * gpr) * 4;
      const size_t q = (size_t)b * RP + (size_t)(y0 + yl) * P + x0;
      float u0[4], u1[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float2 gv = *reinterpret_cast<const float2*>(g1 + (q + j) * 64 + n0);
        if (g2) {
          const float2 g2v = *reinterpret_cast<const float2*>(g2 + (q + j) * 64 + n0);
          gv.x += g2v.x; gv.y += g2v.y;
        }
        u0[j] = gv.x; u1[j] = gv.y;
        accb[0] += gv.x; accb[1] += gv.y;
      }
#pragma unroll
      for (int c = 0; c < CS; ++c)
#pragma unroll
        for (int ty = 0; ty < 3; ++ty) {   // tap (ty, tx) reads the input at (y + ty - 1, x + tx - 1) = smem (yl + ty, x + tx)
          const float* dr = s_x + (c * (kBandRows + 2) + yl + ty) * SW + x0;
          const float2 d01 = *reinterpret_cast<const float2*>(dr);
          const float2 d23 = *reinterpret_cast<const float2*>(dr + 2);
          const float2 d45 = *reinterpret_cast<const float2*>(dr + 4);
          const float d6[6] = {d01.x, d01.y, d23.x, d23.y, d45.x, d45.y};
#pragma unroll
          for (int tx = 0; tx < 3; ++tx)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              acc[0][c * 9 + ty * 3 + tx] = fmaf(u0[j], d6[j + tx], acc[0][c * 9 + ty * 3 + tx]);
              acc[1][c * 9 + ty * 3 + tx] = fmaf(u1[j], d6[j + tx], acc[1][c * 9 + ty * 3 + tx]);
            }
        }
    }
  }
  __syncthreads();
  float* red = s_x;  // [8 warps][64 n][kSwAcc]
#pragma unroll
  for (int j = 0; j < 2; ++j) {
#pragma unroll
    for (int i = 0; i < CS * 9; ++i) red[(wrp * 64 + n0 + j) * kSwAcc + i] = acc[j][i];
    for (int i = CS * 9; i < kSwAcc - 1; ++i) red[(wrp * 64 + n0 + j) * kSwAcc + i] = 0.f;
    red[(wrp * 64 + n0 + j) * kSwAcc + kSwAcc - 1] = accb[j];
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 64 * kSwAcc; i += 256) {
    float sum = 0.f;
#pragma unroll
    for (int ww = 0; ww < 8; ++ww) sum += red[ww * 64 * kSwAcc + i];
    part[(size_t)blockIdx.x * 64 * kSwAcc + i] = sum;
  }
}

__global__ void small_in_wgrad_reduce_kernel(const float* __restrict__ part, int nparts, int Cs, int Ctot, int c0,
                                             float* __restrict__ dw, float* __restrict__ db, int accumulate) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 64 * kSwAcc) return;
  float s = 0.f;
  for (int p = 0; p < nparts; ++p) s += part[(size_t)p * 64 * kSwAcc + i];
  const int n = i / kSwAcc, e = i % kSwAcc;
  if (e == kSwAcc - 1) {
    if (db) db[n] = accumulate ? db[n] + s : s;
  } else if (e < Cs * 9) {
    float* o = dw + (size_t)n * Ctot * 9 + c0 * 9 + e;
    *o = accumulate ? *o + s : s;
  }
}

// ---------------------------------------------------------------------------------------------
// tail-conv weight gradient: dW[c][k][t] = sum_q dout[c][q] * U[q+off(t)][k],  db[c] = sum_q dout[c][q]
// Looping over the rows p of U and scattering to the 9 taps reads U once:
//   dW[c][k][t] += U[p][k] * dout[c][p - off(t)].
// A block owns bands of kBandRows image rows: the planar dout band (+halo, zero outside) is staged in
// shared memory; a thread owns 2 input features k (one bf16x2 load per U row, a warp reads one full
// 128-byte row) and 8 warps walk the band's rows.  Per-block partials, then a fixed-order reduce.
// One launch covers CS <= kChunkC channels c0 .. c0+CS-1 of an output gradient with Ctot channels.
// ---------------------------------------------------------------------------------------------
template <int CS>
__global__ void __launch_bounds__(256, 2)
small_out_wgrad_kernel(const float* __restrict__ dout, const uint16_t* __restrict__ u, int B, int Ctot, int c0, int H,
                       int W, float* __restrict__ part) {
  extern __shared__ float s_buf[];  // 2 x [CS][kBandRows+2][S+2] (column strips, see strip_cols), then the cross-warp reduction buffer
  const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
  const int k0 = lane * 2;
  const int P = W + 1, RP = (H + 1) * P;
  const int S = strip_cols(W), nstrips = (W + S - 1) / S, SWp = S + 2;   // even pitch: 8-byte aligned pairs
  // With 4 image channels a thread's 2 x 36 accumulators (as 64-bit pairs) do not fit 128 registers beside the operands
  // (ptxas kept them in local memory across the loop), so the warps split the channels: even warps take channels 0-1, odd
  // warps 2-3, and each pair of warps walks the same positions (the second read of a U row hits L1).
  constexpr int kSplit = CS > 3 ? 2 : 1, CL = CS / kSplit, kWalkers = 8 / kSplit;
  const int c_lo = kSplit == 2 ? (wrp & 1) * CL : 0, walker = kSplit == 2 ? wrp >> 1 : wrp;
  const bool sums_bias = kSplit == 1 || (wrp & 1) == 0;
  float2 acc[CL * 9];   // .x / .y = the thread's two input features: packed FMAs (ffma2_bcast)
  float accb = 0.f;  // bias gradient: lanes < CS sum channel `lane`
#pragma unroll
  for (int i = 0; i < CL * 9; ++i) acc[i] = make_float2(0.f, 0.f);
  const int bands = (H + kBandRows - 1) / kBandRows;
  const int n_items = B * bands * nstrips, buf_floats = CS * (kBandRows + 2) * SWp;
  if ((int)blockIdx.x < n_items) {
    const BandItem it = band_item(blockIdx.x, bands, nstrips, S);
    stage_band_async(s_buf, dout, CS, Ctot, c0, it.b, H, W, it.y0, it.x_lo, SWp);
  }
  cp_async_commit();
  int parity = 0;
  for (int item = blockIdx.x; item < n_items; item += gridDim.x, parity ^= 1) {
    const BandItem it = band_item(item, bands, nstrips, S);
    const int b = it.b, y0 = it.y0, x_lo = it.x_lo, x_hi = min(W, x_lo + S);
    const float* s_d = s_buf + parity * buf_floats;
    __syncthreads();   // every warp is done with the previous item: its buffer is free for the prefetch
    if (item + (int)gridDim.x < n_items) {
      const BandItem nx = band_item(item + gridDim.x, bands, nstrips, S);
      stage_band_async(s_buf + (parity ^ 1) * buf_floats, dout, CS, Ctot, c0, nx.b, H, W, nx.y0, nx.x_lo, SWp);
    }
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();
    const int rows = min(kBandRows, H - y0);
    const float* s_c = s_d + c_lo * (kBandRows + 2) * SWp;   // this warp's channels
    if ((W & 3) == 0) {
      // four consecutive positions per step: the 6 dout values a 3-tap row needs for them come from three aligned
      // 8-byte shared loads (the pitch is even), 18 loads feed 144 FMAs -- the scalar path below needs 72
      // Rows outside, groups inside (no division per step); the four U rows of the NEXT step are requested before the
      // FMAs of this one -- issued right before their use, the loads were 44 % of the stall samples (ncu, round 2).
      const int ng = (x_hi - x_lo) >> 2;
      for (int yl = 0; yl < rows; ++yl) {
        const uint16_t* urow = u + ((size_t)b * RP + (size_t)(y0 + yl) * P + x_lo) * 64 + k0;
        const float* srow = s_c + yl * SWp;
        uint32_t nxt[4];
        if (walker < ng) {
#pragma unroll
          for (int j = 0; j < 4; ++j) nxt[j] = *reinterpret_cast<const uint32_t*>(urow + (walker * 4 + j) * 64);
        }
        for (int gi = walker; gi < ng; gi += kWalkers) {
          const int xr = gi * 4;
          float2 uu[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) uu[j] = make_float2(bf16_lo(nxt[j]), bf16_hi(nxt[j]));
          if (gi + kWalkers < ng) {
#pragma unroll
            for (int j = 0; j < 4; ++j) nxt[j] = *reinterpret_cast<const uint32_t*>(urow + (xr + kWalkers * 4 + j) * 64);
          }
#pragma unroll
          for (int c = 0; c < CL; ++c)
#pragma unroll
            for (int ry = 0; ry < 3; ++ry) {
              const float* dr = srow + (c * (kBandRows + 2) + ry) * SWp + xr;
              const float2 d01 = *reinterpret_cast<const float2*>(dr);
              const float2 d23 = *reinterpret_cast<const float2*>(dr + 2);
              const float2 d45 = *reinterpret_cast<const float2*>(dr + 4);
              const float d6[6] = {d01.x, d01.y, d23.x, d23.y, d45.x, d45.y};
              const int ty = 2 - ry;   // smem row yl + 2 - ty
#pragma unroll
              for (int tx = 0; tx < 3; ++tx)
#pragma unroll
                for (int j = 0; j < 4; ++j) ffma2_bcast(acc[c * 9 + ty * 3 + tx], uu[j], d6[j + 2 - tx]);
            }
          if (sums_bias && lane < CS) {
            const float* dr = s_d + (lane * (kBandRows + 2) + yl + 1) * SWp + xr + 1;
            accb += (dr[0] + dr[1]) + (dr[2] + dr[3]);
          }
        }
      }
      continue;
    }
    const int ncol = x_hi - x_lo;
    for (int pos = walker; pos < rows * ncol; pos += kWalkers) {
      const int yl = pos / ncol, xr = pos - yl * ncol;
      const size_t q = (size_t)b * RP + (size_t)(y0 + yl) * P + x_lo + xr;
      const uint32_t uv = *reinterpret_cast<const uint32_t*>(u + q * 64 + k0);
      const float2 uu = make_float2(bf16_lo(uv), bf16_hi(uv));
#pragma unroll
      for (int c = 0; c < CL; ++c)
#pragma unroll
        for (int t = 0; t < 9; ++t)
          // output pixel that sees row p through tap t: (y,x) - (t/3-1, t%3-1); smem index shifts by +1 halo
          ffma2_bcast(acc[c * 9 + t], uu, s_c[(c * (kBandRows + 2) + yl + 2 - t / 3) * SWp + xr + 2 - t % 3]);
      if (sums_bias && lane < CS) accb += s_d[(lane * (kBandRows + 2) + yl + 1) * SWp + xr + 1];
    }
  }
  // cross-warp reduction through shared memory: [8 warps][64 k][kSwAcc]; a warp contributes zeros for the channels it
  // does not own
  cp_async_wait<0>();
  __syncthreads();
  float* red = s_buf;
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    float* mine = red + (wrp * 64 + k0 + j) * kSwAcc;
    for (int i = 0; i < kSwAcc; ++i) mine[i] = 0.f;
#pragma unroll
    for (int i = 0; i < CL * 9; ++i) mine[c_lo * 9 + i] = j ? acc[i].y : acc[i].x;
  }
  __syncthreads();
  if (lane < CS) red[(wrp * 64 + lane) * kSwAcc + kSwAcc - 1] = accb;
  __syncthreads();
  for (int i = threadIdx.x; i < 64 * kSwAcc; i += 256) {
    float sum = 0.f;
#pragma unroll
    for (int ww = 0; ww < 8; ++ww) sum += red[ww * 64 * kSwAcc + i];
    part[(size_t)blockIdx.x * 64 * kSwAcc + i] = sum;
  }
}

__global__ void small_out_wgrad_reduce_kernel(const float* __restrict__ part, int nparts, int Cs, int c0,
                                              float* __restrict__ dw, float* __restrict__ db, int accumulate) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 64 * kSwAcc) return;
  float s = 0.f;
  for (int p = 0; p < nparts; ++p) s += part[(size_t)p * 64 * kSwAcc + i];
  const int k = i / kSwAcc, e = i % kSwAcc;
  if (e == kSwAcc - 1) {
    if (db && k < Cs) db[c0 + k] = accumulate ? db[c0 + k] + s : s;
  } else if (e < Cs * 9) {
    const int c = c0 + e / 9, t = e % 9;
    float* o = dw + ((size_t)c * 64 + k) * 9 + t;
    *o = accumulate ? *o + s : s;
  }
}

// ---------------------------------------------------------------------------------------------
// tail conv forward on CUDA cores: 64-feature bf16 PTL -> planar fp32 (B,Cs,H,W).  Used when the image is too
// wide for the tensor-core kernel's flat halo window (W > ~700: the x8 up-scaling of 96x96 tiles); the op is
// HBM-bound either way (it reads 128 B per pixel and writes 4*Cs).  One warp per output pixel: lanes split
// the 64 input features (2 each), 9 taps, shuffle reduction.  One launch writes CS <= kChunkC output planes
// c0 .. c0+CS-1 of Ctot.
// ---------------------------------------------------------------------------------------------
template <int CS>
__global__ void __launch_bounds__(256)
small_out_fwd_kernel(const uint16_t* __restrict__ u, const float* __restrict__ w, const float* __restrict__ bias, int B,
                     int Ctot, int c0, int H, int W, float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  float wr[CS][9][2];
#pragma unroll
  for (int c = 0; c < CS; ++c)
#pragma unroll
    for (int t = 0; t < 9; ++t) {
      wr[c][t][0] = w[((c0 + c) * 64 + 2 * lane) * 9 + t];
      wr[c][t][1] = w[((c0 + c) * 64 + 2 * lane + 1) * 9 + t];
    }
  const int P = W + 1;
  const long long RP = (long long)(H + 1) * P;
  const long long npix = (long long)B * H * W;
  for (long long pix = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); pix < npix; pix += (long long)gridDim.x * 8) {
    const int x = int(pix % W), y = int((pix / W) % H), b = int(pix / ((long long)W * H));
    const long long q = b * RP + (long long)y * P + x;
    float acc[CS];
#pragma unroll
    for (int c = 0; c < CS; ++c) acc[c] = 0.f;
#pragma unroll
    for (int t = 0; t < 9; ++t) {
      const long long qq = q + (t / 3 - 1) * P + (t % 3 - 1);   // padding rows are zero; only the buffer ends need a guard
      if (qq < 0 || qq >= (long long)B * RP) continue;
      const uint32_t v = *reinterpret_cast<const uint32_t*>(u + qq * 64 + 2 * lane);
      const float v0 = bf16_lo(v), v1 = bf16_hi(v);
#pragma unroll
      for (int c = 0; c < CS; ++c) acc[c] = fmaf(wr[c][t][0], v0, fmaf(wr[c][t][1], v1, acc[c]));
    }
#pragma unroll
    for (int c = 0; c < CS; ++c) {
      float a = acc[c];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
      if (lane == 0) out[(((long long)b * Ctot + c0 + c) * H + y) * W + x] = a + (bias ? bias[c0 + c] : 0.f);
    }
  }
}

static int small_grid() {
  int sms = device_sm_count();
  if (sms <= 0) sms = 148;
  return sms * 4;
}

}  // namespace sres

using namespace sres;

extern "C" int sres_conv3x3_small_in(const float* in_nchw, const float* w, const float* bias, int B, int Cs, int H,
                                     int W, int transposed, int unshuffle, float* out_f32, void* out_bf16,
                                     void* stream) {
  if (!in_nchw || !w || (!out_f32 && !out_bf16)) return set_error(SRES_ERR_INVALID_ARG, "small_in: null pointer");
  if (Cs < 1 || Cs > kMaxSmallC) return set_error(SRES_ERR_UNSUPPORTED, "small_in: 1..16 image channels supported");
  if (B <= 0 || H <= 0 || W <= 0) return set_error(SRES_ERR_INVALID_ARG, "small_in: bad geometry");
  if (unshuffle > 1 && (H % unshuffle || W % unshuffle))
    return set_error(SRES_ERR_INVALID_ARG, "small_in: unshuffle factor must divide H and W");
  const int bands = (H + 1 + kBandRows - 1) / kBandRows;
  const bool wide = Cs > kChunkC;
  const int S = wide ? strip_cols_wide(W) : strip_cols(W), nstrips = (W + S - 1) / S;
  long long items = (long long)B * bands * nstrips;
  const int blocks = (int)(items > small_grid() * 2 ? small_grid() * 2 : items);
  cudaStream_t st = (cudaStream_t)stream;
  uint16_t* o16 = (uint16_t*)out_bf16;
  if (wide) {
    const size_t smem = small_in_wide_smem_bytes(Cs, W);   // <= 98.5 KB at 16 channels
    cudaFuncSetAttribute(conv3x3_small_in_wide_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    conv3x3_small_in_wide_kernel<<<blocks, 256, smem, st>>>(in_nchw, w, bias, B, Cs, H, W, transposed, unshuffle, out_f32,
                                                            o16);
    SRES_CHECK_LAUNCH("small_in: launch");
    return SRES_OK;
  }
  const size_t smem = 2 * (size_t)Cs * (kBandRows + 2) * (S + 2) * sizeof(float);   // double buffer, <= 83 KB
#define SRES_LAUNCH_SMALL_IN(CS)                                                                                   \
  do {                                                                                                             \
    if (smem > 48 * 1024)                                                                                          \
      cudaFuncSetAttribute(conv3x3_small_in_kernel<CS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);    \
    conv3x3_small_in_kernel<CS><<<blocks, 256, smem, st>>>(in_nchw, w, bias, B, H, W, transposed, unshuffle, out_f32, o16); \
  } while (0)
  switch (Cs) {
    case 1: SRES_LAUNCH_SMALL_IN(1); break;
    case 2: SRES_LAUNCH_SMALL_IN(2); break;
    case 3: SRES_LAUNCH_SMALL_IN(3); break;
    default: SRES_LAUNCH_SMALL_IN(4); break;
  }
#undef SRES_LAUNCH_SMALL_IN
  SRES_CHECK_LAUNCH("small_in: launch");
  return SRES_OK;
}

// The weight-gradient launches of the channel chunks run one after the other on the caller's stream and reuse the same
// partials, so the workspace is the size of one chunk's, whatever the channel count.
extern "C" size_t sres_small_wgrad_workspace_bytes(void) { return (size_t)small_grid() * 64 * kSwAcc * sizeof(float); }

extern "C" int sres_small_in_wgrad(const float* g1_f32, const float* g2_f32, const float* in_nchw, int B, int Cs,
                                   int H, int W, float* dw, float* db, int accumulate, void* workspace,
                                   size_t workspace_bytes, void* stream) {
  if (!g1_f32 || !in_nchw || !dw || !workspace) return set_error(SRES_ERR_INVALID_ARG, "small_in_wgrad: null pointer");
  if (Cs < 1 || Cs > kMaxSmallC) return set_error(SRES_ERR_UNSUPPORTED, "small_in_wgrad: 1..16 image channels supported");
  const int grid = small_grid();
  if (workspace_bytes < (size_t)grid * 64 * kSwAcc * sizeof(float))
    return set_error(SRES_ERR_INVALID_ARG, "small_in_wgrad: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  float* partp = (float*)workspace;
  // chunks of <= 4 channels; each recomputes the bias gradient, the first one writes it
  for (int c0 = 0; c0 < Cs; c0 += kChunkC) {
    const int cc = Cs - c0 < kChunkC ? Cs - c0 : kChunkC;
    size_t smem = (size_t)cc * (kBandRows + 2) * ((W + 3) & ~1) * sizeof(float);
    const size_t red = (size_t)8 * 64 * kSwAcc * sizeof(float);
    if (smem < red) smem = red;
    if ((W & 3) == 0 && smem <= 200 * 1024) {
#define SRES_LAUNCH_HEAD_WG(CS)                                                                                       \
  do {                                                                                                                \
    cudaFuncSetAttribute(small_in_wgrad_band_kernel<CS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);      \
    small_in_wgrad_band_kernel<CS><<<grid, 256, smem, st>>>(g1_f32, g2_f32, in_nchw, B, Cs, c0, H, W, partp);          \
  } while (0)
      switch (cc) {
        case 1: SRES_LAUNCH_HEAD_WG(1); break;
        case 2: SRES_LAUNCH_HEAD_WG(2); break;
        case 3: SRES_LAUNCH_HEAD_WG(3); break;
        default: SRES_LAUNCH_HEAD_WG(4); break;
      }
#undef SRES_LAUNCH_HEAD_WG
    } else {
      small_in_wgrad_kernel<<<grid, 256, 0, st>>>(g1_f32, g2_f32, in_nchw, B, cc, Cs, c0, H, W, partp);
    }
    SRES_CHECK_LAUNCH("small_in_wgrad: launch");
    small_in_wgrad_reduce_kernel<<<(64 * kSwAcc + 255) / 256, 256, 0, st>>>(partp, grid, cc, Cs, c0, dw,
                                                                             c0 == 0 ? db : nullptr, accumulate);
    SRES_CHECK_LAUNCH("small_in_wgrad: reduce launch");
  }
  return SRES_OK;
}

extern "C" int sres_small_out_wgrad(const float* dout_nchw, const void* u_bf16, int B, int Cs, int H, int W, float* dw,
                                    float* db, int accumulate, void* workspace, size_t workspace_bytes, void* stream) {
  if (!dout_nchw || !u_bf16 || !dw || !workspace) return set_error(SRES_ERR_INVALID_ARG, "small_out_wgrad: null pointer");
  if (Cs < 1 || Cs > kMaxSmallC) return set_error(SRES_ERR_UNSUPPORTED, "small_out_wgrad: 1..16 image channels supported");
  const int grid = small_grid();
  if (workspace_bytes < (size_t)grid * 64 * kSwAcc * sizeof(float))
    return set_error(SRES_ERR_INVALID_ARG, "small_out_wgrad: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  const uint16_t* u16 = (const uint16_t*)u_bf16;
  float* partp = (float*)workspace;
  // chunks of <= 4 channels: each one reads all of U again (the 64-feature operand), see DESIGN.md section 3.3.  Past 4
  // channels a remainder of 3 runs as 2 + 1: the 3-channel instance keeps 27 accumulator pairs a thread and spills.
  for (int c0 = 0, cc; c0 < Cs; c0 += cc) {
    cc = Cs - c0 < kChunkC ? Cs - c0 : kChunkC;
    if (Cs > kChunkC && cc == 3) cc = 2;
    size_t smem = 2 * (size_t)cc * (kBandRows + 2) * (strip_cols(W) + 2) * sizeof(float);   // double buffer
    const size_t red = (size_t)8 * 64 * kSwAcc * sizeof(float);
    if (smem < red) smem = red;
#define SRES_LAUNCH_SMALL_OUT(CS)                                                                               \
  do {                                                                                                          \
    cudaFuncSetAttribute(small_out_wgrad_kernel<CS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);   \
    small_out_wgrad_kernel<CS><<<grid, 256, smem, st>>>(dout_nchw, u16, B, Cs, c0, H, W, partp);                \
  } while (0)
    switch (cc) {
      case 1: SRES_LAUNCH_SMALL_OUT(1); break;
      case 2: SRES_LAUNCH_SMALL_OUT(2); break;
      case 3: SRES_LAUNCH_SMALL_OUT(3); break;
      default: SRES_LAUNCH_SMALL_OUT(4); break;
    }
#undef SRES_LAUNCH_SMALL_OUT
    SRES_CHECK_LAUNCH("small_out_wgrad: launch");
    small_out_wgrad_reduce_kernel<<<(64 * kSwAcc + 255) / 256, 256, 0, st>>>(partp, grid, cc, c0, dw, db, accumulate);
    SRES_CHECK_LAUNCH("small_out_wgrad: reduce launch");
  }
  return SRES_OK;
}

extern "C" int sres_conv3x3_small_out(const void* u_bf16, const float* w, const float* bias, int B, int Cs, int H, int W,
                                      float* out_nchw, void* stream) {
  if (!u_bf16 || !w || !out_nchw) return set_error(SRES_ERR_INVALID_ARG, "small_out: null pointer");
  if (Cs < 1 || Cs > kMaxSmallC) return set_error(SRES_ERR_UNSUPPORTED, "small_out: 1..16 image channels supported");
  if (B <= 0 || H <= 0 || W <= 0) return set_error(SRES_ERR_INVALID_ARG, "small_out: bad geometry");
  const int grid = small_grid() * 4;
  cudaStream_t st = (cudaStream_t)stream;
  const uint16_t* u16 = (const uint16_t*)u_bf16;
  for (int c0 = 0; c0 < Cs; c0 += kChunkC) {   // output planes in chunks of <= 4
    const int cc = Cs - c0 < kChunkC ? Cs - c0 : kChunkC;
    switch (cc) {
      case 1: small_out_fwd_kernel<1><<<grid, 256, 0, st>>>(u16, w, bias, B, Cs, c0, H, W, out_nchw); break;
      case 2: small_out_fwd_kernel<2><<<grid, 256, 0, st>>>(u16, w, bias, B, Cs, c0, H, W, out_nchw); break;
      case 3: small_out_fwd_kernel<3><<<grid, 256, 0, st>>>(u16, w, bias, B, Cs, c0, H, W, out_nchw); break;
      default: small_out_fwd_kernel<4><<<grid, 256, 0, st>>>(u16, w, bias, B, Cs, c0, H, W, out_nchw); break;
    }
    SRES_CHECK_LAUNCH("small_out: launch");
  }
  return SRES_OK;
}
