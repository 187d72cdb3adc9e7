// Two dependent 3x3 convolutions 64 -> 64 in ONE persistent launch (sm_100a): the conv1 -> conv2 pair of an RCAB's forward
// pass and the dgrad(conv2) -> dgrad(conv1) pair of its backward pass.
//
// A single convolution launch (conv_igemm.cu) walks 1201 tiles with 148 CTAs: 17 CTAs own a ninth tile while 131 idle,
// and every launch pays its own pipeline fill (barriers, TMEM, 72 KB of weights, the first halo window, the first tile's
// MMAs with nothing to overlap) and drain (the last tile's epilogue) -- together about a third of the kernel.  The second
// convolution of a pair needs, for its tile t, only tiles t-1, t, t+1 of the first (the halo is P+1 <= 128 rows), and with
// round-robin tile ownership those were finished eight tile-times earlier.  So here every CTA runs its phase-1 tiles and goes
// straight on with its phase-2 tiles (the phase-2 weights have their own region -- PairParams::dual_w, forward pair, see
// pair_slot -- or are swapped in once phase 1's MMAs have retired) -- ownership reversed (CTA c takes tile G-1-c + kG), so that
// the CTAs that owned nine tiles in phase 1 own eight in phase 2: 17 tile-times instead of 18, and ONE fill / drain.
//
// Hand-over through global memory: phase-1 epilogue warps TMA-store their slab of tile t and bump ready[t] once that bulk
// group is COMPLETE (not just its shared-memory reads).  Waiting for completion right away would stall the epilogue, so the
// publication trails the stores by kLag bulk groups (cp.async.bulk.wait_group kLag-1; the tail is flushed after the last
// tile).  The phase-2 TMA producer polls ready[t-1..t+1] == 8 on three lanes in parallel and then loads the halo window
// (protocol variants: fence_proxy_async_mode below).  The counters clean themselves: the last of the (up to three) phase-2
// tiles that consumed ready[t] resets it -- bookkeeping deferred by one tile so it is off the critical path -- so the
// buffer (zero-filled once with the workspace) is ready for the next launch.  All CTAs are co-resident (grid <=
// number of SMs, one CTA per SM), so the waits cannot deadlock; a CTA delayed by another stream's kernel delays its
// neighbours' phase 2 by exactly the time it would have delayed the end of the kernel anyway.
//
// Pipeline, warp roles, shared-memory layout and epilogue code are those of conv_igemm.cu's specialised single-CTA
// instances (tap-per-MMA, 4 TMEM stages, TMA-staged epilogue slabs, fragment-layout column sums).
//
// Replaces two nn.Conv2d(64, 64, 3, padding=1) of the reference per launch
// (sres/model/common/cnn.py:8-9 as used in RCAB, sres/model/rcan/network.py:50-64, and their autograd).
#include "ptx.cuh"
#include "internal.h"
#include "conv_epi.cuh"

namespace sres {

constexpr int kPStages = 6;
constexpr int kPAcc = 4;
constexpr int kPThreads = 384;
constexpr int kPWBytes = 9 * 64 * 128;

struct PairParams {
  int H, W, P, R, npos, n_tiles;
  int nstage, stage_rows, box_rows;
  int off_s16, off_msk, off_s32, off_tail;
  const float* bias1;
  const float* bias2;
  float* part2;            // per-tile partial sums of phase 2 (SRES_EPI_POOL / SRES_EPI_DOT)
  unsigned* ready;         // [n_tiles] phase-1 tiles stored (counts epilogue warps), self-cleaning
  unsigned* consumed;      // [n_tiles] phase-2 tiles that have seen ready[t]
  long long* timeline;     // bring-up only: per-CTA clock stamps [grid][16]
  int strict;              // hand-over protocol: 1 acquire / release with proxy fences, 0 light (see fence_handover)
  int dual_w;              // 0: one 72 KB weight region, swapped between the phases; 1: two regions, and the one a phase does
                           // not need lends its space to the halo ring (see pair_slot)
};

constexpr int kPO16 = 1, kPO32 = 2, kPR32 = 4, kPMsk = 8, kPRelu = 16, kPPool = 32, kPDot = 64;

__device__ __forceinline__ unsigned ld_acquire_gpu(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void red_release_gpu_add(unsigned* p, unsigned v) {
  asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void red_relaxed_gpu_add(unsigned* p, unsigned v) {
  asm volatile("red.relaxed.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned ld_relaxed_gpu(const unsigned* p) {
  unsigned v;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// Hand-over protocol (SRES_PAIR_FENCE=1 selects the strict one):
//   light (default): the tile counter is bumped with red.relaxed.gpu after cp.async.bulk.wait_group has reported the slab
//       store COMPLETE, and read with ld.relaxed.gpu; no gpu-scope fences.  Both the slab (TMA store) and its consumer (TMA
//       load) go straight to L2, the point of coherence at gpu scope, and the counter is bumped strictly after the completion
//       of the store it covers, so a consumer that has seen the count cannot read older data.
//   strict: red.release.gpu / ld.acquire.gpu plus fence.proxy.async.global on both sides -- the by-the-book pattern; the
//       per-tile MEMBAR.GPU of the release costs 0.7 ms per training step (27.87 vs 27.0-27.2 ms; unfused 28.20).
// Both protocols are bit-exact against two separate launches in tests/test_gpu_kernels.py::test_conv_pair_equals_two_launches.
__device__ __forceinline__ void fence_handover(int strict) {
  if (strict) asm volatile("fence.proxy.async.global;" ::: "memory");
}

// per-warp epilogue state shared by both phases
struct EpiWarp {
  uint8_t* s16; uint8_t* smk; uint8_t* s32;
  uint64_t* bin;
  int n_in;              // operand loads issued so far (parity of `bin`)
  int wq, half, lane;
};

// One tile of the TMA-staged epilogue in the ROW layout (thread = TMEM lane): bias, ReLU / ReLU-mask, bf16 slab, TMA store.
template <int FL>
__device__ __forceinline__ void epi_rows(const PairParams& p, EpiWarp& w, const float* s_bias, const CUtensorMap* tmO16,
                                         int tile, uint32_t trow) {
  constexpr bool f_msk = FL & kPMsk, f_relu = FL & kPRelu;
  const int lane = w.lane;
  const int row0 = tile * 128 + w.wq * 32;
  const int q = row0 + lane;
  const int RP = p.R * p.P;
  const int b = q / RP;
  const int rem = q - b * RP;
  const int y = rem / p.P;
  const int x = rem - y * p.P;
  const bool pad = (x == p.W) || (y == p.H) || q >= p.npos;
  uint32_t raw[32];
  tmem_ld32(trow, raw);
  tmem_ld_wait();
  if (f_msk) mbar_wait(w.bin, (w.n_in - 1) & 1, 6);
  const int sw3 = (lane >> 1) & 3;
  uint8_t* r16 = w.s16 + lane * 64;
  const uint8_t* rmk = w.smk + lane * 64;
#pragma unroll
  for (int ch = 0; ch < 2; ++ch) {
    const int c0 = w.half * 32 + ch * 16;
    float v[16];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float4 b4 = *reinterpret_cast<const float4*>(s_bias + c0 + 4 * j);
      v[4 * j + 0] = __uint_as_float(raw[ch * 16 + 4 * j + 0]) + b4.x;
      v[4 * j + 1] = __uint_as_float(raw[ch * 16 + 4 * j + 1]) + b4.y;
      v[4 * j + 2] = __uint_as_float(raw[ch * 16 + 4 * j + 2]) + b4.z;
      v[4 * j + 3] = __uint_as_float(raw[ch * 16 + 4 * j + 3]) + b4.w;
    }
    if (f_relu) {
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.f);
    }
    if (f_msk) {
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const uint4 mk = *reinterpret_cast<const uint4*>(rmk + (((ch * 2 + j) ^ sw3) << 4));
        const uint32_t w4[4] = {mk.x, mk.y, mk.z, mk.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          if (!(bf16_lo(w4[e]) > 0.f)) v[8 * j + 2 * e] = 0.f;
          if (!(bf16_hi(w4[e]) > 0.f)) v[8 * j + 2 * e + 1] = 0.f;
        }
      }
    }
    if (pad) {
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] = 0.f;
    }
#pragma unroll
    for (int j = 0; j < 2; ++j)
      *reinterpret_cast<uint4*>(r16 + (((ch * 2 + j) ^ sw3) << 4)) =
          make_uint4(pack_bf16x2(v[8 * j], v[8 * j + 1]), pack_bf16x2(v[8 * j + 2], v[8 * j + 3]),
                     pack_bf16x2(v[8 * j + 4], v[8 * j + 5]), pack_bf16x2(v[8 * j + 6], v[8 * j + 7]));
  }
  (void)tmO16;
}

// One tile of the fragment-layout epilogue (thread = rows frq + 8j x column pairs 8k + 2fm): bias, fp32 addend, per-tile
// column sums (CA pool / sum g*t2), bf16 and/or fp32 slab.
template <int FL>
__device__ __forceinline__ void epi_frag(const PairParams& p, EpiWarp& w, const float (&bias8)[8], int tile, uint32_t trow) {
  constexpr bool f_o16 = FL & kPO16, f_o32 = FL & kPO32, f_r32 = FL & kPR32, f_msk = FL & kPMsk, f_dot = FL & kPDot;
  constexpr bool use_in = f_msk || f_r32;
  const int lane = w.lane;
  const int fm = lane & 3, frq = lane >> 2;
  const int fcol = ((lane >> 4) & 1) * 16 + ((lane >> 3) & 1) * 8 + 2 * fm + ((lane >> 2) & 1);
  const int row0 = tile * 128 + w.wq * 32;
  const int q = row0 + lane;
  const int RP = p.R * p.P;
  const int b = q / RP;
  const int rem = q - b * RP;
  const int y = rem / p.P;
  const int x = rem - y * p.P;
  const bool pad = (x == p.W) || (y == p.H) || q >= p.npos;
  const int seg = (b != (tile * 128) / RP) ? 1 : 0;
  uint32_t fa[16], fb[16];
  tmem_ld_frag16(trow, fa);
  tmem_ld_frag16(trow + (16u << 16), fb);
  const unsigned padmask = __ballot_sync(0xffffffffu, pad);
  const unsigned seg1 = __ballot_sync(0xffffffffu, seg == 1);
  const bool mixed = seg1 != 0u && seg1 != 0xffffffffu;
  tmem_ld_wait();
  if (use_in) mbar_wait(w.bin, (w.n_in - 1) & 1, 6);
  const int sw3 = (frq >> 1) & 3;
  float cs0[8], cs1[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) cs0[i] = cs1[i] = 0.f;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int r = frq + 8 * j;
    const bool rpad = (padmask >> r) & 1u;
    const bool rs1 = (seg1 >> r) & 1u;
    uint8_t* row32 = w.s32 + r * 128 + (fm & 1) * 8;
    uint8_t* row16 = w.s16 + r * 64 + 4 * fm;
    const uint8_t* rowmk = w.smk + r * 64 + 4 * fm;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const uint32_t* src = (j < 2) ? fa : fb;
      float v0 = __uint_as_float(src[4 * k + 2 * (j & 1)]) + bias8[2 * k];
      float v1 = __uint_as_float(src[4 * k + 2 * (j & 1) + 1]) + bias8[2 * k + 1];
      const int o32 = ((2 * k + (fm >> 1)) ^ frq) << 4;
      const int o16 = (k ^ sw3) << 4;
      if (f_r32) {
        const float2 rr = *reinterpret_cast<const float2*>(row32 + o32);
        v0 += rr.x; v1 += rr.y;
      }
      uint32_t mk = 0;
      if (f_msk) mk = *reinterpret_cast<const uint32_t*>(rowmk + o16);
      if (f_msk && !f_dot) {
        if (!(bf16_lo(mk) > 0.f)) v0 = 0.f;
        if (!(bf16_hi(mk) > 0.f)) v1 = 0.f;
      }
      if (rpad) { v0 = 0.f; v1 = 0.f; }
      float c0v = v0, c1v = v1;
      if (f_dot) { c0v = v0 * bf16_lo(mk); c1v = v1 * bf16_hi(mk); }
      if (mixed && rs1) { cs1[2 * k] += c0v; cs1[2 * k + 1] += c1v; }
      else { cs0[2 * k] += c0v; cs0[2 * k + 1] += c1v; }
      if (f_o32) *reinterpret_cast<float2*>(row32 + o32) = make_float2(v0, v1);
      if (f_o16) *reinterpret_cast<uint32_t*>(row16 + o16) = pack_bf16x2(v0, v1);
    }
  }
  const float t0 = frag_colsum(cs0, lane);
  const float t1 = mixed ? frag_colsum(cs1, lane) : 0.f;
  float* dst = p.part2 + ((long long)tile * 2 * 4 + w.wq) * 64 + w.half * 32 + fcol;
  const bool all1 = seg1 == 0xffffffffu;
  dst[0] = all1 ? 0.f : t0;
  dst[4 * 64] = all1 ? t0 : t1;
}

// Which halo-ring slot the i-th tile of a phase uses, and how often that slot has been used before (mbarrier parity).
//
// One weight region (dual_w 0): slot = it % nstage over the whole launch.
//
// Lending mode (dual_w 1, the forward pair): with both 72 KB weight regions the ring has only two slots of its own (B0, B1) --
// one tile of prefetch, and the MMA warp waited for TMA 10 % of the time.  But phase 1 does not need the phase-2 weights'
// region and phase 2 does not need phase 1's, and a region holds two slots: phase 1 cycles through X0 X1 B0 B1 (X in the
// phase-2 weight region) for all but its last two tiles, which use B0 B1 only; once X0 / X1 are released for the last time
// the phase-2 weights are loaded there, two tile-times before they are needed.  Phase 2 starts on B0 B1 and, from its third
// tile on, cycles B0 B1 Y0 Y1 (Y in the phase-1 weight region, free once the last phase-1 MMA has retired -- which the
// producer has seen by then: it waited for B1's release by the last phase-1 tile).  Physical slots: 0 1 = B, 2 3 = X, 4 5 = Y.
// (The sequence and the use counts below were checked on the host against a running count for every n1, n2 < 60.)
struct SlotUse { int slot; uint32_t use; };
__device__ __forceinline__ SlotUse pair_slot(int lend, int nstage, int phase, int i, int it, int n1) {
  if (!lend) return SlotUse{it % nstage, uint32_t(it / nstage)};
  if (phase == 0) {
    if (i >= n1 - 2) {
      const int sl = i - (n1 - 2);                                        // B0 (if n1 >= 2), then B1
      return SlotUse{sl, uint32_t((n1 - 2 + sl) / 4)};
    }
    const int m = (n1 - 3 - i) & 3;                                        // distance from the last lent tile
    return SlotUse{m == 0 ? 3 : m == 1 ? 2 : m == 2 ? 1 : 0, uint32_t(i >> 2)};
  }
  const int m = i & 3;
  const uint32_t b0 = n1 >= 2 ? uint32_t((n1 - 2) / 4 + 1) : 0u, b1 = n1 >= 1 ? uint32_t((n1 - 1) / 4 + 1) : 0u;   // phase-1 uses
  return SlotUse{m == 0 ? 0 : m == 1 ? 1 : m == 2 ? 4 : 5, uint32_t(i >> 2) + (m == 0 ? b0 : m == 1 ? b1 : 0u)};
}

template <int FL1, int FL2>
__global__ void __launch_bounds__(kPThreads, 1)
conv3x3_pair_kernel(const __grid_constant__ CUtensorMap tmA1, const __grid_constant__ CUtensorMap tmW1,
                    const __grid_constant__ CUtensorMap tmO1, const __grid_constant__ CUtensorMap tmM1,
                    const __grid_constant__ CUtensorMap tmA2, const __grid_constant__ CUtensorMap tmW2,
                    const __grid_constant__ CUtensorMap tmO16_2, const __grid_constant__ CUtensorMap tmM2,
                    const __grid_constant__ CUtensorMap tmR32_2, const __grid_constant__ CUtensorMap tmO32_2,
                    const PairParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* smem_w = smem;
  uint8_t* smem_w2 = smem + (p.dual_w ? kPWBytes : 0);
  uint8_t* smem_a = smem + kPWBytes * (p.dual_w ? 2 : 1);
  const int stage_bytes = p.stage_rows * 128;
  // byte offset of a physical ring slot from smem_a (slots 2..5 exist in lending mode only and lie in the weight regions)
  auto slot_off = [&](int slot) -> int {
    if (slot < 2 || !p.dual_w) return slot * stage_bytes;
    return (slot < 4 ? kPWBytes + (slot - 2) * stage_bytes : (slot - 4) * stage_bytes) - 2 * kPWBytes;
  };
  uint8_t* tail = smem + p.off_tail;
  uint64_t* bar_full = reinterpret_cast<uint64_t*>(tail);   // [kPStages]
  uint64_t* bar_empty = bar_full + kPStages;                // [kPStages]
  uint64_t* bar_w = bar_empty + kPStages;                   // [2] weights of phase 1 / phase 2
  uint64_t* bar_tfull = bar_w + 2;                          // [kPAcc]
  uint64_t* bar_tempty = bar_tfull + kPAcc;                 // [kPAcc]
  uint64_t* bar_in = bar_tempty + kPAcc;                    // [8]
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(bar_in + 8);
  float* s_bias = reinterpret_cast<float*>(tmem_holder + 4);  // [2][64], 16-byte aligned (float4 loads)

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  const int G = gridDim.x;
  const int c1 = blockIdx.x;             // phase-1 tiles: c1 + kG
  const int c2 = G - 1 - blockIdx.x;     // phase-2 tiles: c2 + kG (reversed ownership balances the ninth tiles)
  const int n1 = c1 < p.n_tiles ? (p.n_tiles - 1 - c1) / G + 1 : 0;
  long long* tl = p.timeline ? p.timeline + (size_t)blockIdx.x * 16 : nullptr;
#define PSTAMP(i)                              \
  do {                                         \
    if (tl && lane == 0) tl[i] = clock64();    \
  } while (0)
  if (tl && threadIdx.x == 0) { tl[0] = clock64(); tl[12] = tl[13] = tl[14] = tl[15] = 0; }

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmA1);
    tma_prefetch_desc(&tmW1);
    tma_prefetch_desc(&tmA2);
    tma_prefetch_desc(&tmW2);
    for (int i = 0; i < kPStages; ++i) {
      mbar_init(&bar_full[i], 1);
      mbar_init(&bar_empty[i], 1);
    }
    mbar_init(&bar_w[0], 1);
    mbar_init(&bar_w[1], 1);
    for (int i = 0; i < kPAcc; ++i) {
      mbar_init(&bar_tfull[i], 1);
      mbar_init(&bar_tempty[i], 8);
    }
    for (int i = 0; i < 8; ++i) mbar_init(&bar_in[i], 1);
    mbar_fence_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_holder, kPAcc * 64);
    tmem_relinquish();
  }
  if (threadIdx.x < 64) s_bias[threadIdx.x] = p.bias1 ? p.bias1[threadIdx.x] : 0.f;
  else if (threadIdx.x < 128) s_bias[threadIdx.x] = p.bias2 ? p.bias2[threadIdx.x - 64] : 0.f;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_holder, 0);
  if (warp == 0) PSTAMP(1);
  pdl_launch_dependents();

  if (warp == 0) {
    // ===================== TMA producer =====================
    const bool leader = elect_one();
    if (leader) {
      mbar_expect_tx(&bar_w[0], kPWBytes);
      for (int t = 0; t < 9; ++t) tma_load_2d(smem_w + t * 64 * 128, &tmW1, &bar_w[0], 0, t * 64);
    }
    pdl_wait();
    int it = 0;
    for (int tile = c1; tile < p.n_tiles; tile += G, ++it) {
      const SlotUse su = pair_slot(p.dual_w, p.nstage, 0, it, it, n1);
      const int slot = su.slot;
      const uint32_t ph = su.use & 1;
      mbar_wait(&bar_empty[slot], ph ^ 1, 1);
      const int row0 = tile * 128 - (p.P + 1);
      uint8_t* dst = smem_a + slot_off(slot);
      if (leader) {
        mbar_expect_tx(&bar_full[slot], stage_bytes);
        for (int r = 0; r < p.stage_rows; r += p.box_rows) tma_load_2d(dst + r * 128, &tmA1, &bar_full[slot], 0, row0 + r);
      }
      __syncwarp();
    }
    if (p.dual_w) {
      // lending mode: the phase-2 weights go where the lent slots X0 / X1 were, once phase 1 has released them for the last
      // time (X0 was used n1 / 4 times, X1 (n1 + 1) / 4 times) -- its last two tiles are still running on B0 / B1
      const int ux0 = n1 / 4, ux1 = (n1 + 1) / 4;
      if (ux0 > 0) mbar_wait(&bar_empty[2], uint32_t(ux0 - 1) & 1, 7);
      if (ux1 > 0) mbar_wait(&bar_empty[3], uint32_t(ux1 - 1) & 1, 7);
      PSTAMP(2);   // lent slots released
      if (leader) {
        mbar_expect_tx(&bar_w[1], kPWBytes);
        for (int t = 0; t < 9; ++t) tma_load_2d(smem_w2 + t * 64 * 128, &tmW2, &bar_w[1], 0, t * 64);
      }
      __syncwarp();
    } else {
      // phase-2 weights replace phase 1's once every phase-1 MMA of this CTA has retired (its last ring slot was released)
      if (n1 > 0) mbar_wait(&bar_empty[(n1 - 1) % p.nstage], ((n1 - 1) / p.nstage) & 1, 7);
      PSTAMP(2);   // every phase-1 MMA retired
      if (leader) {
        mbar_expect_tx(&bar_w[1], kPWBytes);
        for (int t = 0; t < 9; ++t) tma_load_2d(smem_w + t * 64 * 128, &tmW2, &bar_w[1], 0, t * 64);
      }
      __syncwarp();
    }
    // Lanes 0..2 watch one phase-1 tile each (t-1, t, t+1 cover this tile's halo window: P + 1 <= 128 rows).  The counters
    // clean themselves -- the last of the (up to three) phase-2 tiles that has seen ready[t] resets it -- and that
    // bookkeeping runs one tile behind, its atomic in flight while the lane spins on the next counter, so the producer stays
    // ahead of the tensor core (the first version did six dependent global round trips per tile on one lane and made
    // phase 2 producer-bound: +14 us per launch).
    int prev_t = -1;          // the phase-1 tile this lane watched for the previous phase-2 tile
    for (int tile = c2, i2 = 0; tile < p.n_tiles; tile += G, ++it, ++i2) {
      // lanes 4..6 watch (never the elected lane: a gpu-scope acquire on the thread that has TMA loads in flight waits for
      // those loads and stops the producer from running ahead of the tensor core)
      const int t = tile - 1 + (lane - 4);
      const bool watch = lane >= 4 && lane < 7 && t >= 0 && t < p.n_tiles;
      unsigned seen = 0;
      long long f0 = 0;
      if (tl) f0 = clock64();
      if (prev_t >= 0) seen = atomicAdd(p.consumed + prev_t, 1u) + 1u;
      if (watch) {
        long long t0 = clock64();
        while ((p.strict ? ld_acquire_gpu(p.ready + t) : ld_relaxed_gpu(p.ready + t)) < 8u) {
          __nanosleep(32);
          if (clock64() - t0 > 8000000000LL) { atomicExch(&g_sres_dev_error, 0xDEAD0008u); __threadfence_system(); __trap(); }
        }
      }
      if (prev_t >= 0) {
        const unsigned users = (prev_t > 0 ? 1u : 0u) + 1u + (prev_t + 1 < p.n_tiles ? 1u : 0u);
        if (seen == users) { p.ready[prev_t] = 0u; p.consumed[prev_t] = 0u; }
      }
      prev_t = watch ? t : -1;
      if (watch) fence_handover(p.strict);   // generic acquire -> async-proxy reads, on a lane without TMA ops in flight
      __syncwarp();
      if (tl && lane == 4) tl[12] += clock64() - f0;   // producer: flag bookkeeping + spinning, phase 2
      // (the watchers' acquires and proxy fences are ordered before the elected lane's TMA load by the warp barrier above;
      // the elected lane itself issues no fence: it would wait for its own TMA loads in flight)
      const SlotUse su = pair_slot(p.dual_w, p.nstage, 1, i2, it, n1);
      const int slot = su.slot;
      const uint32_t ph = su.use & 1;
      mbar_wait(&bar_empty[slot], ph ^ 1, 1);
      const int row0 = tile * 128 - (p.P + 1);
      uint8_t* dst = smem_a + slot_off(slot);
      if (leader) {
        mbar_expect_tx(&bar_full[slot], stage_bytes);
        for (int r = 0; r < p.stage_rows; r += p.box_rows) tma_load_2d(dst + r * 128, &tmA2, &bar_full[slot], 0, row0 + r);
      }
      __syncwarp();
    }
    if (prev_t >= 0) {
      const unsigned users = (prev_t > 0 ? 1u : 0u) + 1u + (prev_t + 1 < p.n_tiles ? 1u : 0u);
      if (atomicAdd(p.consumed + prev_t, 1u) + 1u == users) { p.ready[prev_t] = 0u; p.consumed[prev_t] = 0u; }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    const bool leader = elect_one();
    constexpr uint32_t idesc = make_idesc_bf16(128, 64, 0, 0);
    constexpr uint32_t dhi = sdesc_hi_sw128(1024);
    uint32_t w_lo = sdesc_lo(smem_u32(smem_w), 16);
    const uint32_t a_lo0 = sdesc_lo(smem_u32(smem_a), 16);
    const uint32_t row_step = uint32_t(p.P) * 8;
    int it = 0;
#pragma unroll 1
    for (int phase = 0; phase < 2; ++phase) {
      mbar_wait(&bar_w[phase], 0, 2);
      tc_fence_after();
      if (phase == 1) w_lo = sdesc_lo(smem_u32(smem_w2), 16);
      PSTAMP(3 + 3 * phase);   // weights of this phase landed
      for (int tile = phase ? c2 : c1, ip = 0; tile < p.n_tiles; tile += G, ++it, ++ip) {
        const SlotUse su = pair_slot(p.dual_w, p.nstage, phase, ip, it, n1);
        const int slot = su.slot;
        const uint32_t ph = su.use & 1;
        const int acc = it % kPAcc;
        const uint32_t aph = (it / kPAcc) & 1;
        long long w0 = 0, w1 = 0;
        if (tl) w0 = clock64();
        mbar_wait(&bar_tempty[acc], aph ^ 1, 3);
        if (tl) w1 = clock64();
        mbar_wait(&bar_full[slot], ph, 4);
        if (tl && lane == 0) { tl[14] += w1 - w0; tl[15] += clock64() - w1; }   // MMA warp waiting for the epilogue / for TMA
        tc_fence_after();
        const uint32_t a_tile = p.dual_w ? sdesc_lo(smem_u32(smem_a) + slot_off(slot), 16) : a_lo0 + uint32_t(slot * stage_bytes) / 16;
        const uint32_t d_tmem = tmem_base + uint32_t(acc * 64);
        if (leader) {
#pragma unroll
          for (int t = 0; t < 9; ++t) {
            const uint32_t a_tap = a_tile + uint32_t(t / 3) * row_step + uint32_t(t % 3) * 8;
            const uint32_t b_tap = w_lo + uint32_t(t * 64 * 8);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              if (t == 0 && k == 0) umma_bf16_lohi<false>(d_tmem, a_tap, dhi, b_tap, dhi, idesc);
              else umma_bf16_lohi<true>(d_tmem, a_tap + k * 2, dhi, b_tap + k * 2, dhi, idesc);
            }
          }
          umma_commit(&bar_empty[slot]);
          umma_commit(&bar_tfull[acc]);
        }
        __syncwarp();
      }
      PSTAMP(4 + 3 * phase);   // last MMA of this phase issued
    }
  } else if (warp >= 4) {
    // ===================== epilogue =====================
    EpiWarp w;
    const int ew = warp - 4;
    w.wq = warp & 3; w.half = ew >> 2; w.lane = lane; w.n_in = 0;
    w.s16 = smem + p.off_s16 + ew * 2048;
    w.smk = smem + p.off_msk + ew * 2048;
    w.s32 = smem + p.off_s32 + ew * 4096;
    w.bin = &bar_in[ew];
    constexpr bool in1 = FL1 & kPMsk;
    constexpr bool in2 = (FL2 & kPMsk) || (FL2 & kPR32);
    pdl_wait();
    int it = 0;
    // Phase-1 tiles whose slab store has been issued but not yet published.  A store is published once its bulk group has
    // COMPLETED (global writes done; about 3500 cycles after issue under load): waiting for a young group stalls the epilogue
    // and, through the TMA unit, the halo loads (kLag = 3: +4000 cycles per phase).  So up to kLag groups stay in flight and a
    // tile is published kLag tiles after its store was issued -- early enough, because phase 2 needs wave k of phase 1 only at
    // its own wave k; only the slab's shared-memory READS are awaited every tile.
    constexpr int kLag = 5;
    int pend[kLag];
#pragma unroll
    for (int i = 0; i < kLag; ++i) pend[i] = -1;
    // ---------------- phase 1 ----------------
    for (int tile = c1; tile < p.n_tiles; tile += G, ++it) {
      const int acc = it % kPAcc;
      const uint32_t aph = (it / kPAcc) & 1;
      const int row0 = tile * 128 + w.wq * 32;
      if (lane == 0) {
        bulk_wait_read<0>();                        // the slab may be overwritten
        if (pend[0] >= 0) {
          bulk_wait_all<kLag - 1>();                 // the oldest pending store has reached global memory ...
          fence_handover(p.strict);                  // (async-proxy writes ordered before the generic release)
          if (p.strict) red_release_gpu_add(p.ready + pend[0], 1u);
          else red_relaxed_gpu_add(p.ready + pend[0], 1u);   // ... publish it to the phase-2 producers of other CTAs
        }
        if (in1) {
          mbar_expect_tx(w.bin, 2048u);
          tma_load_2d(w.smk, &tmM1, w.bin, w.half * 32, row0);
        }
      }
      if (in1) ++w.n_in;
      __syncwarp();
      mbar_wait(&bar_tfull[acc], aph, 5);
      tc_fence_after();
      const uint32_t trow = tmem_base + (uint32_t(w.wq * 32) << 16) + uint32_t(acc * 64 + w.half * 32);
      epi_rows<FL1>(p, w, s_bias, &tmO1, tile, trow);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_tempty[acc]);
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        tma_store_2d(&tmO1, w.s16, w.half * 32, row0);
        bulk_commit();
      }
#pragma unroll
      for (int i = 0; i + 1 < kLag; ++i) pend[i] = pend[i + 1];
      pend[kLag - 1] = tile;
    }
    if (lane == 0) {
      bulk_wait_all<0>();
      fence_handover(p.strict);
#pragma unroll
      for (int i = 0; i < kLag; ++i)
        if (pend[i] >= 0) {
          if (p.strict) red_release_gpu_add(p.ready + pend[i], 1u);
          else red_relaxed_gpu_add(p.ready + pend[i], 1u);
        }
    }
    __syncwarp();
    if (warp == 4) PSTAMP(5);   // phase-1 epilogue done, all tiles published
    // ---------------- phase 2 ----------------
    const int fm = lane & 3;
    float bias8[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) bias8[i] = s_bias[64 + w.half * 32 + 8 * (i >> 1) + 2 * fm + (i & 1)];
    for (int tile = c2; tile < p.n_tiles; tile += G, ++it) {
      const int acc = it % kPAcc;
      const uint32_t aph = (it / kPAcc) & 1;
      const int row0 = tile * 128 + w.wq * 32;
      if (lane == 0) {
        bulk_wait_read<0>();
        if (in2) {
          mbar_expect_tx(w.bin, ((FL2 & kPMsk) ? 2048u : 0u) + ((FL2 & kPR32) ? 4096u : 0u));
          if (FL2 & kPMsk) tma_load_2d(w.smk, &tmM2, w.bin, w.half * 32, row0);
          if (FL2 & kPR32) tma_load_2d(w.s32, &tmR32_2, w.bin, w.half * 32, row0);
        }
      }
      if (in2) ++w.n_in;
      __syncwarp();
      mbar_wait(&bar_tfull[acc], aph, 5);
      tc_fence_after();
      const uint32_t trow = tmem_base + (uint32_t(w.wq * 32) << 16) + uint32_t(acc * 64 + w.half * 32);
      epi_frag<FL2>(p, w, bias8, tile, trow);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_tempty[acc]);
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        if (FL2 & kPO16) tma_store_2d(&tmO16_2, w.s16, w.half * 32, row0);
        if (FL2 & kPO32) tma_store_2d(&tmO32_2, w.s32, w.half * 32, row0);
        bulk_commit();
      }
    }
    if (lane == 0) bulk_wait_all<0>();
    if (warp == 4) PSTAMP(8);   // phase-2 epilogue done
  }

  tc_fence_before();
  __syncthreads();
  if (tl && threadIdx.x == 0) tl[9] = clock64();
  if (warp == 2) tmem_dealloc(tmem_base, kPAcc * 64);
#undef PSTAMP
}

// shared-memory plan of a pair launch; false when the halo ring would have fewer than two slots
static bool pair_plan(int W, bool fwd, PairParams* p, size_t* smem_bytes) {
  const int smem_max = 232448;
  const int slab = fwd ? 16384 : (16384 + 16384 + 32768);   // bf16 out | bf16 out + mask + fp32 read-modify-write
  const int rows = 128 + 2 * (W + 2);
  const int box = (rows + 7) / 8 * 8 <= 256 ? (rows + 7) / 8 * 8 : 64;   // the whole window as one TMA box when it fits
  const int stage_rows = (rows + box - 1) / box * box;
  // Two weight regions when that still leaves a ring of two slots or more (stages of <= 260 rows for the forward pair).  The
  // region a phase does not need then lends the ring two more slots (pair_slot): a 72 KB region holds two stages of <= 288 rows.
  const bool dual = (smem_max - 1024 - 2 * kPWBytes - 1024 - slab) / (stage_rows * 128) >= 2;
  int ns = dual ? 2 : (smem_max - 1024 - kPWBytes - 1024 - slab) / (stage_rows * 128);
  if (ns > kPStages) ns = kPStages;
  if (ns < 2) return false;
  if (p) {
    p->box_rows = box; p->stage_rows = stage_rows; p->nstage = ns; p->dual_w = dual ? 1 : 0;
    int off = kPWBytes * (dual ? 2 : 1) + ns * stage_rows * 128;   // (lending mode: 2 ring slots of its own, 4 more inside the weight regions)
    p->off_s16 = off; off += 16384;
    p->off_msk = off; off += fwd ? 0 : 16384;
    p->off_s32 = off; off += fwd ? 0 : 32768;
    p->off_tail = off; off += 1024;
    *smem_bytes = (size_t)off + 1024;
  }
  return true;
}

static bool conv_pair_fuse_enabled() {
  static const int on = [] {
    const char* e = getenv("SRES_CONV_FUSE");
    return e ? atoi(e) : 1;
  }();
  return on != 0;
}

}  // namespace sres

using namespace sres;

extern "C" size_t sres_conv_pair_flag_bytes(int B, int H, int W) {
  const long long npos = (long long)B * (H + 1) * (W + 1);
  return (size_t)((npos + 127) / 128) * 2 * sizeof(unsigned);
}

// 1 when the (first, second) convolution flavours and the geometry can run as one fused launch
extern "C" int sres_conv_pair_supported(const sres_conv_args* a1, const sres_conv_args* a2) {
  if (!conv_pair_fuse_enabled() || !a1 || !a2) return 0;
  if (a1->B != a2->B || a1->H != a2->H || a1->W != a2->W || a1->W + 2 > 128) return 0;
  if (a1->n_out != 64 || a2->n_out != 64 || a1->map_mode != SRES_MAP_IDENT || a2->map_mode != SRES_MAP_IDENT) return 0;
  if (a1->out_bf16 == nullptr || a2->in_bf16 != a1->out_bf16) return 0;
  if (a1->out_f32 || a1->resid_f32 || a1->resid2_f32 || a1->out_nchw || a2->resid2_f32 || a2->out_nchw) return 0;
  if (a1->debug_flags || a2->debug_flags) return 0;
  const long long npos = (long long)a1->B * (a1->H + 1) * (a1->W + 1);
  if ((a1->H + 1) * (a1->W + 1) < 128 || npos > 0x7fffff00LL) return 0;
  const bool fwd = (a1->epi_flags == SRES_EPI_RELU) && !a1->mask_bf16 && a2->epi_flags == SRES_EPI_POOL && a2->out_bf16 &&
                   !a2->out_f32 && !a2->resid_f32 && !a2->mask_bf16 && a2->pool_part;
  const bool bwd = a1->epi_flags == 0 && a1->mask_bf16 && a2->epi_flags == SRES_EPI_DOT && a2->mask_bf16 && a2->out_f32 &&
                   a2->resid_f32 && !a2->out_bf16 && a2->pool_part;
  return ((fwd || bwd) && pair_plan(a1->W, fwd, nullptr, nullptr)) ? 1 : 0;
}

extern "C" int sres_conv3x3_pair(const sres_conv_args* a1, const sres_conv_args* a2, void* flags, void* stream_) {
  if (!sres_conv_pair_supported(a1, a2) || !flags) return set_error(SRES_ERR_UNSUPPORTED, "conv pair: flavours / geometry not fusable");
  cudaStream_t stream = (cudaStream_t)stream_;
  const bool fwd = a1->epi_flags == SRES_EPI_RELU;
  PairParams p{};
  p.H = a1->H; p.W = a1->W; p.P = a1->W + 1; p.R = a1->H + 1;
  p.npos = (int)((long long)a1->B * p.R * p.P);
  p.n_tiles = (p.npos + 127) / 128;
  p.bias1 = a1->bias; p.bias2 = a2->bias; p.part2 = a2->pool_part;
  p.ready = (unsigned*)flags; p.consumed = p.ready + p.n_tiles;
  p.timeline = (long long*)a1->debug_timeline;
  {
    static const int strict = [] { const char* e = getenv("SRES_PAIR_FENCE"); return e && atoi(e) == 1 ? 1 : 0; }();
    p.strict = strict;
  }
  const int smem_max = 232448;
  size_t smem = 0;
  if (!pair_plan(a1->W, fwd, &p, &smem)) return set_error(SRES_ERR_UNSUPPORTED, "conv pair: no room for the halo ring");

  CUtensorMap tmA1, tmW1, tmO1, tmM1, tmA2, tmW2, tmO16_2, tmM2, tmR32_2, tmO32_2;
  int rc;
  if ((rc = make_tmap_rows64(&tmA1, a1->in_bf16, (uint64_t)p.npos, p.box_rows))) return rc;
  if ((rc = make_tmap_rows64(&tmW1, a1->wpack_bf16, 9 * 64, 64))) return rc;
  if ((rc = make_tmap_rows64_half(&tmO1, a1->out_bf16, (uint64_t)p.npos, 32))) return rc;
  tmM1 = tmO1;
  if (a1->mask_bf16 && (rc = make_tmap_rows64_half(&tmM1, a1->mask_bf16, (uint64_t)p.npos, 32))) return rc;
  if ((rc = make_tmap_rows64(&tmA2, a2->in_bf16, (uint64_t)p.npos, p.box_rows))) return rc;
  if ((rc = make_tmap_rows64(&tmW2, a2->wpack_bf16, 9 * 64, 64))) return rc;
  tmO16_2 = tmO1; tmM2 = tmO1; tmR32_2 = tmO1; tmO32_2 = tmO1;
  if (a2->out_bf16 && (rc = make_tmap_rows64_half(&tmO16_2, a2->out_bf16, (uint64_t)p.npos, 32))) return rc;
  if (a2->mask_bf16 && (rc = make_tmap_rows64_half(&tmM2, a2->mask_bf16, (uint64_t)p.npos, 32))) return rc;
  if (a2->resid_f32 && (rc = make_tmap_rows64_f32(&tmR32_2, a2->resid_f32, (uint64_t)p.npos, 32))) return rc;
  if (a2->out_f32 && (rc = make_tmap_rows64_f32(&tmO32_2, a2->out_f32, (uint64_t)p.npos, 32))) return rc;

  const int sms = device_sm_count();
  if (sms <= 0) return set_error(SRES_ERR_NO_DEVICE, "conv pair: no CUDA device");
  const int grid = p.n_tiles < sms ? p.n_tiles : sms;
  int dev = 0;
  cudaGetDevice(&dev);
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(kPThreads); cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  cudaError_t e;
  if (fwd) {
    auto k = conv3x3_pair_kernel<kPRelu | kPO16, kPPool | kPO16>;
    static thread_local int attr_dev = -1;
    if (attr_dev != dev) {
      if ((e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max)) != cudaSuccess) return set_cuda_error(e, "conv pair: smem attribute");
      attr_dev = dev;
    }
    count_launch();
    e = cudaLaunchKernelEx(&cfg, k, tmA1, tmW1, tmO1, tmM1, tmA2, tmW2, tmO16_2, tmM2, tmR32_2, tmO32_2, p);
  } else {
    auto k = conv3x3_pair_kernel<kPMsk | kPO16, kPR32 | kPO32 | kPMsk | kPDot>;
    static thread_local int attr_dev = -1;
    if (attr_dev != dev) {
      if ((e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max)) != cudaSuccess) return set_cuda_error(e, "conv pair: smem attribute");
      attr_dev = dev;
    }
    count_launch();
    e = cudaLaunchKernelEx(&cfg, k, tmA1, tmW1, tmO1, tmM1, tmA2, tmW2, tmO16_2, tmM2, tmR32_2, tmO32_2, p);
  }
  if (e != cudaSuccess) return set_cuda_error(e, "conv pair: launch");
  e = cudaGetLastError();
  if (e != cudaSuccess) return set_cuda_error(e, "conv pair: launch");
  return SRES_OK;
}
