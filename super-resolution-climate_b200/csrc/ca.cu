// Channel attention (CALayer) + RCAB residual, forward and backward, on the padded tile layout.
// Memory-bound: every kernel touches each 64-channel row with 16/32-byte vector accesses, one
// 8-channel slice per thread, and the tiny squeeze-excite MLP is recomputed per block.
//
// Reference: sres/model/rcan/network.py:31-47 (CALayer: AdaptiveAvgPool2d(1) -> 1x1 conv F->F/r ->
// ReLU -> 1x1 conv F/r->F -> Sigmoid -> x*y) and :61-64 (RCAB: res = body(x); res += x).
#include "internal.h"
#include "ptx.cuh"

namespace sres {

constexpr int kCaThreads = 256;
constexpr int kCaMaxHidden = 64;

struct CaGeom {
  int B, H, W, P, RP;   // RP = (H+1)*(W+1)
  int hid;              // F / reduction
  int blocks_per_image;
  int tile_rows;        // output rows per M tile of the convolution that wrote the per-tile partial sums (126 or 128)
};

// ---- shared: s = sigmoid(W2 relu(W1 m + b1) + b2) for one image -----------------------------
// sm_m[64] must hold the pooled means.  Fills sm_h[hid], sm_z[64], sm_s[64].  All 256 threads call.
// Each output is one warp-wide dot product (coalesced weight rows + shuffle reduce), 8 warps in parallel:
// the chain is latency-bound, so it must be short -- it sits between two full-tensor passes.
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ void ca_mlp(const float* __restrict__ w1, const float* __restrict__ b1,
                                       const float* __restrict__ w2, const float* __restrict__ b2, int hid,
                                       const float* sm_m, float* sm_h, float* sm_z, float* sm_s) {
  const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
  const float m0 = sm_m[lane], m1 = sm_m[lane + 32];
  for (int j = wrp; j < hid; j += kCaThreads / 32) {
    const float v = warp_sum(fmaf(__ldg(w1 + j * 64 + lane), m0, __ldg(w1 + j * 64 + 32 + lane) * m1));
    if (lane == 0) sm_h[j] = fmaxf(v + __ldg(b1 + j), 0.f);
  }
  __syncthreads();
  for (int c = wrp; c < 64; c += kCaThreads / 32) {
    float v = lane < hid ? __ldg(w2 + c * hid + lane) * sm_h[lane] : 0.f;
    if (lane + 32 < hid) v = fmaf(__ldg(w2 + c * hid + lane + 32), sm_h[lane + 32], v);
    v = warp_sum(v);
    if (lane == 0) {
      const float z = v + __ldg(b2 + c);
      sm_z[c] = z;
      sm_s[c] = 1.f / (1.f + expf(-z));
    }
  }
  __syncthreads();
}

// ---- the same MLP with the weights staged in shared memory -----------------------------------
// The apply kernels sit between two tensor-core kernels and every block repeats the pooled-mean -> MLP chain, so
// its latency is paid once per RCAB per direction.  Staging the four small parameter arrays with ONE round of global
// loads (issued together with the loads of the per-tile partial sums) leaves only shared-memory phases in the chain.
struct CaWeights {
  float* w1;   // [hid][64]
  float* w2t;  // [hid][64] (transposed: conflict-free for both products)
  float* b1;   // [hid]
  float* b2;   // [64]
};
static size_t ca_weights_bytes(int hid) { return (size_t)(2 * hid * 64 + hid + 64) * sizeof(float); }
__device__ __forceinline__ void ca_stage_weights(CaWeights& S, const float* __restrict__ w1, const float* __restrict__ b1,
                                                 const float* __restrict__ w2, const float* __restrict__ b2, int hid) {
  extern __shared__ float ca_dyn_smem[];
  S.w1 = ca_dyn_smem; S.w2t = S.w1 + hid * 64; S.b1 = S.w2t + hid * 64; S.b2 = S.b1 + hid;
  for (int i = threadIdx.x; i < hid * 64; i += kCaThreads) {
    S.w1[i] = __ldg(w1 + i);
    S.w2t[(i % hid) * 64 + i / hid] = __ldg(w2 + i);
  }
  if (threadIdx.x < hid) S.b1[threadIdx.x] = __ldg(b1 + threadIdx.x);
  if (threadIdx.x < 64) S.b2[threadIdx.x] = __ldg(b2 + threadIdx.x);
}
// h = relu(W1 m + b1): one warp per hidden unit.  Caller syncs before (sm_m, weights) and after.
__device__ __forceinline__ void ca_hidden(const CaWeights& S, int hid, const float* sm_m, float* sm_h) {
  const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
  const float m0 = sm_m[lane], m1 = sm_m[lane + 32];
  for (int j = wrp; j < hid; j += kCaThreads / 32) {
    const float v = warp_sum(fmaf(S.w1[j * 64 + lane], m0, S.w1[j * 64 + 32 + lane] * m1));
    if (lane == 0) sm_h[j] = fmaxf(v + S.b1[j], 0.f);
  }
}
// z = W2 h + b2 and s = sigmoid(z) for channel c = threadIdx.x < 64
__device__ __forceinline__ float ca_logit(const CaWeights& S, int hid, const float* sm_h, int c) {
  float z = S.b2[c];
  for (int j = 0; j < hid; ++j) z = fmaf(S.w2t[j * 64 + c], sm_h[j], z);
  return z;
}
__device__ __forceinline__ float ca_gate(const CaWeights& S, int hid, const float* sm_h, int c) {
  return 1.f / (1.f + expf(-ca_logit(S, hid, sm_h, c)));
}
// sigmoid'(z) = s (1 - s) with 1 - s = sigmoid(-z): 1.f - s cancels where s nears 1 (z = 9: 4e-4 relative error, and 0
// from z = 17 on, where s rounds to 1)
__device__ __forceinline__ float ca_dsigmoid(float s, float z) { return s / (1.f + expf(z)); }

// ---- stand-alone average-pool sums (used when an image is smaller than one 128-row M tile, where
// the conv epilogue's two-segment partials do not apply) --------------------------------------
__global__ void __launch_bounds__(kCaThreads)
ca_pool_kernel(CaGeom g, const uint16_t* __restrict__ t2, float* __restrict__ pool_sum) {
  __shared__ float sm[kCaThreads / 8][64 + 1];
  const int b = blockIdx.x, tid = threadIdx.x, cg = tid & 7;
  float a[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (int r = tid >> 3; r < g.RP; r += kCaThreads / 8) {
    const uint4 tv = *reinterpret_cast<const uint4*>(t2 + ((size_t)b * g.RP + r) * 64 + cg * 8);
    a[0] += bf16_lo(tv.x); a[1] += bf16_hi(tv.x); a[2] += bf16_lo(tv.y); a[3] += bf16_hi(tv.y);
    a[4] += bf16_lo(tv.z); a[5] += bf16_hi(tv.z); a[6] += bf16_lo(tv.w); a[7] += bf16_hi(tv.w);
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) sm[tid >> 3][cg * 8 + j] = a[j];
  __syncthreads();
  if (tid < 64) {
    float s = 0.f;
    for (int i = 0; i < kCaThreads / 8; ++i) s += sm[i][tid];
    pool_sum[b * 64 + tid] = s;
  }
}

// ---- forward --------------------------------------------------------------------------------
// x_out = x_in + t2 * s ;  xb_out = bf16(x_out) ; block 0 of each image stores mean and s.
// Low register count on purpose: all blocks of the grid must be co-resident (one wave), otherwise every
// wave pays the latency-bound pooled-mean + MLP prologue again.
__global__ void __launch_bounds__(kCaThreads)
ca_apply_fwd_kernel(CaGeom g, const uint16_t* __restrict__ t2, const float* __restrict__ pool_part,
                    const float* __restrict__ pool_sum, const float* __restrict__ w1, const float* __restrict__ b1,
                    const float* __restrict__ w2, const float* __restrict__ b2, const float* x_in, float* x_out,
                    uint16_t* __restrict__ xb_out, float* __restrict__ save_mean, float* __restrict__ save_s) {
  __shared__ float sm_red[4][64];
  __shared__ float sm_m[64], sm_h[kCaMaxHidden], sm_s[64];
  CaWeights sw;
  const int b = blockIdx.y, tid = threadIdx.x;
  const int cg = tid & 7;  // 8-channel slice
  ca_stage_weights(sw, w1, b1, w2, b2, g.hid);  // parameters are not written by the previous kernel
  pdl_wait();
  pdl_launch_dependents();
  const int per_blk = (g.RP + g.blocks_per_image - 1) / g.blocks_per_image;
  const int r0 = blockIdx.x * per_blk + (tid >> 3), r1 = min(g.RP, blockIdx.x * per_blk + per_blk);
  // pooled mean from the conv epilogue partials: tiles covering rows [b*RP, (b+1)*RP)
  if (pool_sum) {
    sm_red[tid >> 6][tid & 63] = (tid < 64) ? pool_sum[b * 64 + tid] : 0.f;
  } else {
    const int c = tid & 63, part = tid >> 6;  // 4 partial sums per channel
    const int t0 = (b * g.RP) / g.tile_rows, t1 = ((b + 1) * g.RP - 1) / g.tile_rows;
    float a = 0.f;
#pragma unroll 8
    for (int t = t0; t <= t1; ++t) {
      const int seg = (t * g.tile_rows >= b * g.RP) ? 0 : 1;  // a tile that starts in the previous image holds this one as segment 1
      a += pool_part[(((size_t)t * 2 + seg) * 4 + part) * 64 + c];
    }
    sm_red[part][c] = a;
  }
  __syncthreads();
  if (tid < 64) sm_m[tid] = (sm_red[0][tid] + sm_red[1][tid] + sm_red[2][tid] + sm_red[3][tid]) / float(g.H * g.W);
  __syncthreads();
  ca_hidden(sw, g.hid, sm_m, sm_h);
  __syncthreads();
  if (tid < 64) {
    const float sg = ca_gate(sw, g.hid, sm_h, tid);
    sm_s[tid] = sg;
    if (blockIdx.x == 0) {
      save_mean[b * 64 + tid] = sm_m[tid];
      save_s[b * 64 + tid] = sg;
    }
  }
  __syncthreads();
  // A thread owns channels [4cg, 4cg+4) and [32+4cg, 32+4cg+4): every load/store instruction of a warp then
  // covers whole contiguous 128-byte (fp32) / 64-byte (bf16) row halves -- fully coalesced per instruction.
  float s8[8];
#pragma unroll
  for (int j = 0; j < 4; ++j) { s8[j] = sm_s[cg * 4 + j]; s8[4 + j] = sm_s[32 + cg * 4 + j]; }
#pragma unroll 2
  for (int r = r0; r < r1; r += kCaThreads / 8) {
    const size_t q = (size_t)b * g.RP + r;
    const uint2 ta = *reinterpret_cast<const uint2*>(t2 + q * 64 + cg * 4);
    const uint2 tb = *reinterpret_cast<const uint2*>(t2 + q * 64 + 32 + cg * 4);
    const float4 xa = *reinterpret_cast<const float4*>(x_in + q * 64 + cg * 4);
    const float4 xb = *reinterpret_cast<const float4*>(x_in + q * 64 + 32 + cg * 4);
    float o[8];
    o[0] = fmaf(bf16_lo(ta.x), s8[0], xa.x); o[1] = fmaf(bf16_hi(ta.x), s8[1], xa.y);
    o[2] = fmaf(bf16_lo(ta.y), s8[2], xa.z); o[3] = fmaf(bf16_hi(ta.y), s8[3], xa.w);
    o[4] = fmaf(bf16_lo(tb.x), s8[4], xb.x); o[5] = fmaf(bf16_hi(tb.x), s8[5], xb.y);
    o[6] = fmaf(bf16_lo(tb.y), s8[6], xb.z); o[7] = fmaf(bf16_hi(tb.y), s8[7], xb.w);
    *reinterpret_cast<float4*>(x_out + q * 64 + cg * 4) = make_float4(o[0], o[1], o[2], o[3]);
    *reinterpret_cast<float4*>(x_out + q * 64 + 32 + cg * 4) = make_float4(o[4], o[5], o[6], o[7]);
    if (xb_out) {
      *reinterpret_cast<uint2*>(xb_out + q * 64 + cg * 4) = make_uint2(pack_bf16x2(o[0], o[1]), pack_bf16x2(o[2], o[3]));
      *reinterpret_cast<uint2*>(xb_out + q * 64 + 32 + cg * 4) = make_uint2(pack_bf16x2(o[4], o[5]), pack_bf16x2(o[6], o[7]));
    }
  }
}

// ---- backward, pass 1: ds[b][c] partials = sum_q g[q][c] * t2[q][c] --------------------------
__global__ void __launch_bounds__(kCaThreads)
ca_bwd_reduce_kernel(CaGeom g, const float* __restrict__ grad, const uint16_t* __restrict__ t2,
                     float* __restrict__ ds_part) {
  __shared__ float sm[kCaThreads / 8][64 + 1];
  pdl_wait();
  pdl_launch_dependents();
  const int b = blockIdx.y, tid = threadIdx.x, cg = tid & 7;
  const int per_blk = (g.RP + g.blocks_per_image - 1) / g.blocks_per_image;
  const int r0 = blockIdx.x * per_blk, r1 = min(g.RP, r0 + per_blk);
  float a[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (int r = r0 + (tid >> 3); r < r1; r += kCaThreads / 8) {
    const size_t q = (size_t)b * g.RP + r;
    const uint2 ta = *reinterpret_cast<const uint2*>(t2 + q * 64 + cg * 4);
    const uint2 tb = *reinterpret_cast<const uint2*>(t2 + q * 64 + 32 + cg * 4);
    const float4 ga = *reinterpret_cast<const float4*>(grad + q * 64 + cg * 4);
    const float4 gb = *reinterpret_cast<const float4*>(grad + q * 64 + 32 + cg * 4);
    a[0] = fmaf(ga.x, bf16_lo(ta.x), a[0]); a[1] = fmaf(ga.y, bf16_hi(ta.x), a[1]);
    a[2] = fmaf(ga.z, bf16_lo(ta.y), a[2]); a[3] = fmaf(ga.w, bf16_hi(ta.y), a[3]);
    a[4] = fmaf(gb.x, bf16_lo(tb.x), a[4]); a[5] = fmaf(gb.y, bf16_hi(tb.x), a[5]);
    a[6] = fmaf(gb.z, bf16_lo(tb.y), a[6]); a[7] = fmaf(gb.w, bf16_hi(tb.y), a[7]);
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) { sm[tid >> 3][cg * 4 + j] = a[j]; sm[tid >> 3][32 + cg * 4 + j] = a[4 + j]; }
  __syncthreads();
  if (tid < 64) {
    float s = 0.f;
    for (int i = 0; i < kCaThreads / 8; ++i) s += sm[i][tid];
    ds_part[((size_t)b * g.blocks_per_image + blockIdx.x) * 64 + tid] = s;
  }
}

// ---- backward, pass 2: dt2 = g*s + dm/(H*W) (bf16), padding rows stay 0 ----------------------
__global__ void __launch_bounds__(kCaThreads)
ca_bwd_apply_kernel(CaGeom g, const float* __restrict__ grad, const float* __restrict__ ds_part,
                    const float* __restrict__ tile_part, const float* __restrict__ w1, const float* __restrict__ b1, const float* __restrict__ w2,
                    const float* __restrict__ b2, const float* __restrict__ save_mean,
                    uint16_t* __restrict__ dt2, float* __restrict__ save_ds) {
  __shared__ float sm_m[64], sm_h[kCaMaxHidden], sm_s[64], sm_dz[64], sm_dh[kCaMaxHidden], sm_dm[64];
  __shared__ float sm_dsr[4][64];
  CaWeights sw;
  const int b = blockIdx.y, tid = threadIdx.x;
  const int lane = tid & 31, wrp = tid >> 5, cg = tid & 7;
  ca_stage_weights(sw, w1, b1, w2, b2, g.hid);
  pdl_wait();
  pdl_launch_dependents();
  const int per_blk = (g.RP + g.blocks_per_image - 1) / g.blocks_per_image;
  const int r0 = blockIdx.x * per_blk + (tid >> 3), r1 = min(g.RP, blockIdx.x * per_blk + per_blk);
  if (tile_part) {  // ds was reduced per M tile by the producing convolution (SRES_EPI_DOT)
    const int c = tid & 63, part = tid >> 6;
    const int t0 = (b * g.RP) / g.tile_rows, t1 = ((b + 1) * g.RP - 1) / g.tile_rows;
    float a = 0.f;
#pragma unroll 8
    for (int t = t0; t <= t1; ++t) {
      const int seg = (t * g.tile_rows >= b * g.RP) ? 0 : 1;
      a += tile_part[(((size_t)t * 2 + seg) * 4 + part) * 64 + c];
    }
    sm_dsr[part][c] = a;
  } else if (tid < 64) {
    float a = 0.f;
    for (int i = 0; i < g.blocks_per_image; ++i) a += ds_part[((size_t)b * g.blocks_per_image + i) * 64 + tid];
    sm_dsr[0][tid] = a;
    sm_dsr[1][tid] = sm_dsr[2][tid] = sm_dsr[3][tid] = 0.f;
  }
  if (tid < 64) sm_m[tid] = save_mean[b * 64 + tid];
  __syncthreads();
  ca_hidden(sw, g.hid, sm_m, sm_h);
  __syncthreads();
  if (tid < 64) {
    const float ds = (sm_dsr[0][tid] + sm_dsr[1][tid]) + (sm_dsr[2][tid] + sm_dsr[3][tid]);
    if (blockIdx.x == 0) save_ds[b * 64 + tid] = ds;
    const float z = ca_logit(sw, g.hid, sm_h, tid);
    const float sg = 1.f / (1.f + expf(-z));
    sm_s[tid] = sg;
    sm_dz[tid] = ds * ca_dsigmoid(sg, z);
  }
  __syncthreads();
  // dh[j] = relu'(h[j]) * sum_c w2[c][j] dz[c]: one warp per hidden unit
  for (int j = wrp; j < g.hid; j += kCaThreads / 32) {
    const float v = warp_sum(fmaf(sw.w2t[j * 64 + lane], sm_dz[lane], sw.w2t[j * 64 + 32 + lane] * sm_dz[lane + 32]));
    if (lane == 0) sm_dh[j] = sm_h[j] > 0.f ? v : 0.f;
  }
  __syncthreads();
  if (tid < 64) {  // dm[c] = sum_j w1[j][c] dh[j] / (H*W)
    float a = 0.f;
    for (int j = 0; j < g.hid; ++j) a = fmaf(sw.w1[j * 64 + tid], sm_dh[j], a);
    sm_dm[tid] = a / float(g.H * g.W);
  }
  __syncthreads();
  float s8[8], m8[8];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    s8[j] = sm_s[cg * 4 + j]; s8[4 + j] = sm_s[32 + cg * 4 + j];
    m8[j] = sm_dm[cg * 4 + j]; m8[4 + j] = sm_dm[32 + cg * 4 + j];
  }
  int y = r0 / g.P, x = r0 - y * g.P;
  // Loads are unconditional (padding rows are ordinary readable rows) and the padding test is a select, so the
  // unrolled loop issues all its loads up front: with the loads under a branch only 32 B per thread were in flight
  // and the pass was latency-bound (4.2 TB/s L2-warm).
#pragma unroll 4
  for (int r = r0; r < r1; r += kCaThreads / 8) {
    const size_t q = (size_t)b * g.RP + r;
    const float4 ga = *reinterpret_cast<const float4*>(grad + q * 64 + cg * 4);
    const float4 gb = *reinterpret_cast<const float4*>(grad + q * 64 + 32 + cg * 4);
    const bool valid = (x != g.W) && (y != g.H);
    uint2 oa, ob;
    oa.x = pack_bf16x2(fmaf(ga.x, s8[0], m8[0]), fmaf(ga.y, s8[1], m8[1]));
    oa.y = pack_bf16x2(fmaf(ga.z, s8[2], m8[2]), fmaf(ga.w, s8[3], m8[3]));
    ob.x = pack_bf16x2(fmaf(gb.x, s8[4], m8[4]), fmaf(gb.y, s8[5], m8[5]));
    ob.y = pack_bf16x2(fmaf(gb.z, s8[6], m8[6]), fmaf(gb.w, s8[7], m8[7]));
    if (!valid) { oa = make_uint2(0, 0); ob = make_uint2(0, 0); }
    *reinterpret_cast<uint2*>(dt2 + q * 64 + cg * 4) = oa;
    *reinterpret_cast<uint2*>(dt2 + q * 64 + 32 + cg * 4) = ob;
    x += kCaThreads / 8;
    while (x >= g.P) { x -= g.P; ++y; }
  }
}

// ---- backward: parameter gradients of the squeeze-excite MLP, all RCABs in one launch --------
// One block per CALayer; loops over the batch in a fixed order (deterministic).
struct CaParamBatch {
  const float* params;   // first CALayer's conv_du.0.weight
  float* grads;          // same position in the gradient buffer
  long long layer_stride;  // floats between consecutive CALayers (one RCAB)
  const float* mean;     // [njobs][B][64] saved by forward
  const float* ds;       // [njobs][B][64] saved by backward
};

// pass 1: one block per (layer, image): dz = ds*s*(1-s), h = relu(W1 m + b1), dh = relu'(.) * W2^T dz
__global__ void __launch_bounds__(kCaThreads)
ca_param_prep_kernel(const CaParamBatch batch, int B, int hid, float* __restrict__ scratch) {
  __shared__ float sm_m[64], sm_h[kCaMaxHidden], sm_z[64], sm_s[64], sm_dz[64];
  const int layer = blockIdx.x, b = blockIdx.y, tid = threadIdx.x;
  const long long o = (long long)layer * batch.layer_stride;
  const float* w1 = batch.params + o;
  const float* b1 = w1 + hid * 64;
  const float* w2 = b1 + hid;
  const float* b2 = w2 + 64 * hid;
  if (tid < 64) sm_m[tid] = batch.mean[((size_t)layer * B + b) * 64 + tid];
  __syncthreads();
  ca_mlp(w1, b1, w2, b2, hid, sm_m, sm_h, sm_z, sm_s);
  float* out = scratch + ((size_t)layer * B + b) * (64 + 2 * kCaMaxHidden);  // [dz 64][h 64][dh 64]
  if (tid < 64) {
    const float s = sm_s[tid];
    const float dz = batch.ds[((size_t)layer * B + b) * 64 + tid] * ca_dsigmoid(s, sm_z[tid]);
    sm_dz[tid] = dz;
    out[tid] = dz;
  }
  __syncthreads();
  if (tid < hid) {
    float a = 0.f;
    for (int c = 0; c < 64; ++c) a = fmaf(w2[c * hid + tid], sm_dz[c], a);
    out[64 + tid] = sm_h[tid];
    out[64 + kCaMaxHidden + tid] = sm_h[tid] > 0.f ? a : 0.f;
  }
}

// pass 2: one block per layer: outer-product sums over the batch in a fixed order (deterministic).  The per-image vectors
// (dz, h, dh from pass 1 and the pooled mean) are staged in shared memory chunk by chunk with fully parallel, coalesced loads;
// the sums then run out of shared memory.  (The first version walked the batch with dependent global loads: 69 us per
// launch for 20 blocks, 0.7 ms per training step.)
constexpr int kCaParamChunk = 32;   // images per shared-memory chunk: 32 x 256 floats = 32 KB
__global__ void __launch_bounds__(kCaThreads)
ca_param_sum_kernel(const CaParamBatch batch, int B, int hid, const float* __restrict__ scratch, int accumulate) {
  __shared__ float sm[kCaParamChunk][4][64];   // [image][dz | h | dh | mean][64]
  const int layer = blockIdx.x, tid = threadIdx.x;
  const long long o = (long long)layer * batch.layer_stride;
  float* dw1 = batch.grads + o;
  float* db1 = dw1 + hid * 64;
  float* dw2 = db1 + hid;
  float* db2 = dw2 + 64 * hid;
  const int n12 = hid * 64;
  float a1[16], a2[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) a1[i] = a2[i] = 0.f;
  float ab1 = 0.f, ab2 = 0.f;
  for (int b0 = 0; b0 < B; b0 += kCaParamChunk) {
    const int nb = min(kCaParamChunk, B - b0);
    __syncthreads();
    for (int i = tid; i < nb * 256; i += kCaThreads) {
      const int b = i >> 8, k = (i >> 6) & 3, c = i & 63;
      const size_t img = (size_t)layer * B + b0 + b;
      sm[b][k][c] = k < 3 ? scratch[img * (64 + 2 * kCaMaxHidden) + k * 64 + c] : batch.mean[img * 64 + c];
    }
    __syncthreads();
    for (int b = 0; b < nb; ++b) {
      const float* dz = sm[b][0];
      const float* h = sm[b][1];
      const float* dh = sm[b][2];
      const float* m = sm[b][3];
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const int e = tid + i * kCaThreads;
        if (e < n12) {
          a1[i] = fmaf(dh[e / 64], m[e % 64], a1[i]);    // dw1[j][c] = dh[j] * m[c]
          a2[i] = fmaf(dz[e / hid], h[e % hid], a2[i]);  // dw2[c][j] = dz[c] * h[j]
        }
      }
      if (tid < hid) ab1 += dh[tid];
      if (tid < 64) ab2 += dz[tid];
    }
  }
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const int e = tid + i * kCaThreads;
    if (e < n12) {
      dw1[e] = accumulate ? dw1[e] + a1[i] : a1[i];
      dw2[e] = accumulate ? dw2[e] + a2[i] : a2[i];
    }
  }
  if (tid < hid) db1[tid] = accumulate ? db1[tid] + ab1 : ab1;
  if (tid < 64) db2[tid] = accumulate ? db2[tid] + ab2 : ab2;
}

static int ca_geom(CaGeom* g, int B, int H, int W, int hid) {
  if (B <= 0 || H <= 0 || W <= 0) return set_error(SRES_ERR_INVALID_ARG, "ca: bad geometry");
  if (hid < 1 || hid > kCaMaxHidden) return set_error(SRES_ERR_UNSUPPORTED, "ca: hidden width must be 1..64");
  g->B = B; g->H = H; g->W = W; g->P = W + 1; g->RP = (H + 1) * (W + 1); g->hid = hid;
  int sms = device_sm_count();
  if (sms <= 0) sms = 148;
  int bpi = (4 * sms + B - 1) / B;            // ~4 blocks per SM in total: one resident wave
  const int max_bpi = (g->RP + 31) / 32;      // at least one 32-row sweep each
  if (bpi > max_bpi) bpi = max_bpi;
  if (bpi < 1) bpi = 1;
  g->blocks_per_image = bpi;
  g->tile_rows = sres_conv_tile_rows(H, W);
  return SRES_OK;
}

}  // namespace sres

using namespace sres;

extern "C" int sres_ca_blocks_per_image(int B, int H, int W) {
  CaGeom g;
  if (ca_geom(&g, B, H, W, 1)) return -1;
  return g.blocks_per_image;
}

extern "C" int sres_ca_pool(const void* t2_bf16, float* pool_sum, int B, int H, int W, void* stream) {
  CaGeom g;
  int rc = ca_geom(&g, B, H, W, 1);
  if (rc) return rc;
  if (!t2_bf16 || !pool_sum) return set_error(SRES_ERR_INVALID_ARG, "ca_pool: null pointer");
  ca_pool_kernel<<<B, kCaThreads, 0, (cudaStream_t)stream>>>(g, (const uint16_t*)t2_bf16, pool_sum);
  SRES_CHECK_LAUNCH("ca_pool: launch");
  return SRES_OK;
}

extern "C" int sres_ca_apply_fwd(const void* t2_bf16, const float* pool_part, const float* pool_sum, const float* w1, const float* b1,
                                 const float* w2, const float* b2, int hidden, const float* x_in, float* x_out,
                                 void* xb_out_bf16, float* save_mean, float* save_s, int B, int H, int W,
                                 void* stream) {
  CaGeom g;
  int rc = ca_geom(&g, B, H, W, hidden);
  if (rc) return rc;
  if (!pool_sum && g.RP < 128) return set_error(SRES_ERR_UNSUPPORTED, "ca_apply_fwd: fused pool partials need (H+1)*(W+1) >= 128; pass pool_sum");
  if (!t2_bf16 || (!pool_part && !pool_sum) || !w1 || !b1 || !w2 || !b2 || !x_in || !x_out || !save_mean || !save_s)
    return set_error(SRES_ERR_INVALID_ARG, "ca_apply_fwd: null pointer");
  dim3 grid(g.blocks_per_image, B);
  cudaError_t e = launch_pdl_if(pdl_level() >= 2, ca_apply_fwd_kernel, grid, dim3(kCaThreads), ca_weights_bytes(hidden), (cudaStream_t)stream, g, (const uint16_t*)t2_bf16,
                             pool_part, pool_sum, w1, b1, w2, b2, x_in, x_out, (uint16_t*)xb_out_bf16, save_mean, save_s);
  if (e != cudaSuccess) return set_cuda_error(e, "ca_apply_fwd: launch");
  return SRES_OK;
}

extern "C" int sres_ca_bwd(const float* grad_f32, const void* t2_bf16, const float* w1, const float* b1,
                           const float* w2, const float* b2, int hidden, const float* save_mean, float* ds_part,
                           void* dt2_bf16, float* save_ds, int B, int H, int W, void* stream) {
  CaGeom g;
  int rc = ca_geom(&g, B, H, W, hidden);
  if (rc) return rc;
  if (!grad_f32 || !t2_bf16 || !w1 || !b1 || !w2 || !b2 || !save_mean || !ds_part || !dt2_bf16 || !save_ds)
    return set_error(SRES_ERR_INVALID_ARG, "ca_bwd: null pointer");
  dim3 grid(g.blocks_per_image, B);
  cudaError_t e = launch_pdl_if(pdl_level() >= 2, ca_bwd_reduce_kernel, grid, dim3(kCaThreads), 0, (cudaStream_t)stream, g, grad_f32,
                             (const uint16_t*)t2_bf16, ds_part);
  if (e != cudaSuccess) return set_cuda_error(e, "ca_bwd: reduce launch");
  e = launch_pdl_if(pdl_level() >= 2, ca_bwd_apply_kernel, grid, dim3(kCaThreads), ca_weights_bytes(hidden), (cudaStream_t)stream, g, grad_f32, (const float*)ds_part, (const float*)nullptr, w1, b1,
                 w2, b2, save_mean, (uint16_t*)dt2_bf16, save_ds);
  if (e != cudaSuccess) return set_cuda_error(e, "ca_bwd: apply launch");
  return SRES_OK;
}

extern "C" int sres_ca_bwd_apply(const float* grad_f32, const float* tile_part, const float* w1, const float* b1,
                                 const float* w2, const float* b2, int hidden, const float* save_mean, void* dt2_bf16,
                                 float* save_ds, int B, int H, int W, void* stream) {
  CaGeom g;
  int rc = ca_geom(&g, B, H, W, hidden);
  if (rc) return rc;
  if (g.RP < 128) return set_error(SRES_ERR_UNSUPPORTED, "ca_bwd_apply: per-tile partials need (H+1)*(W+1) >= 128");
  if (!grad_f32 || !tile_part || !w1 || !b1 || !w2 || !b2 || !save_mean || !dt2_bf16 || !save_ds)
    return set_error(SRES_ERR_INVALID_ARG, "ca_bwd_apply: null pointer");
  dim3 grid(g.blocks_per_image, B);
  cudaError_t e = launch_pdl_if(pdl_level() >= 2, ca_bwd_apply_kernel, grid, dim3(kCaThreads), ca_weights_bytes(hidden), (cudaStream_t)stream, g, grad_f32,
                                (const float*)nullptr, tile_part, w1, b1, w2, b2, save_mean, (uint16_t*)dt2_bf16, save_ds);
  if (e != cudaSuccess) return set_cuda_error(e, "ca_bwd_apply: launch");
  return SRES_OK;
}

extern "C" size_t sres_ca_param_grads_scratch_bytes(int nlayers, int B) {
  return (size_t)(nlayers > 0 ? nlayers : 0) * (B > 0 ? B : 0) * (64 + 2 * kCaMaxHidden) * sizeof(float);
}

extern "C" int sres_ca_param_grads(const float* params_first, float* grads_first, int64_t layer_stride, int nlayers,
                                   const float* save_mean, const float* save_ds, int B, int hidden, int accumulate,
                                   void* scratch, size_t scratch_bytes, void* stream) {
  if (!params_first || !grads_first || !save_mean || !save_ds || !scratch || nlayers <= 0 || B <= 0)
    return set_error(SRES_ERR_INVALID_ARG, "ca_param_grads: bad argument");
  if (hidden < 1 || hidden > kCaMaxHidden) return set_error(SRES_ERR_UNSUPPORTED, "ca: hidden width must be 1..64");
  if (scratch_bytes < sres_ca_param_grads_scratch_bytes(nlayers, B))
    return set_error(SRES_ERR_INVALID_ARG, "ca_param_grads: scratch too small");
  CaParamBatch batch{params_first, grads_first, (long long)layer_stride, save_mean, save_ds};
  ca_param_prep_kernel<<<dim3(nlayers, B), kCaThreads, 0, (cudaStream_t)stream>>>(batch, B, hidden, (float*)scratch);
  SRES_CHECK_LAUNCH("ca_param_grads: prep launch");
  ca_param_sum_kernel<<<nlayers, kCaThreads, 0, (cudaStream_t)stream>>>(batch, B, hidden, (const float*)scratch, accumulate);
  SRES_CHECK_LAUNCH("ca_param_grads: sum launch");
  return SRES_OK;
}
