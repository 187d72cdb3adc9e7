// 3x3 convolution over the padded tile layout as a tcgen05 implicit GEMM (sm_100a).
//
//   D[q][n] = sum_{tap,k} A[q + off(tap)][k] * Wp[tap][n][k]        q = PTL row, k = 64 in-features
//
// One persistent CTA per SM; the unit of work is one 128-row M tile.  For a tile the TMA producer
// loads ONE halo window of PTL rows [q0 - (P+1), q0 + 128 + (P+1)) into a shared-memory ring slot
// (128B-swizzled rows, out-of-range rows zero-filled by TMA); the 9 taps are UMMA operands taken from
// that single window by shifting the descriptor start address by (ky*P + kx) rows -- the halo is read
// from L2 once, not once per tap.  The packed weights of all 9 taps stay resident in shared memory for
// the life of the CTA.  Accumulators live in TMEM, 4 stages deep, so the eight epilogue warps drain
// tile i while the tensor core works on tiles i+1..i+3.
//
// Epilogue I/O is TMA too when rows map to themselves: every epilogue warp owns a 32-row x 32-channel
// slab in shared memory; fp32 addends and the bf16 ReLU mask are TMA-loaded into it while the MMAs
// run, results are written back into the slab and TMA-stored (full lines, no LSU traffic).
// PixelShuffle-scattered and planar (NCHW) outputs take the direct global-store path.
//
// Warp roles (384 threads): 0 = TMA producer, 1 = MMA issuer, 2 = TMEM allocator, 4..11 = epilogue
// (two warps per TMEM lane quarter, each 32 of the 64 output columns).
//
// Replaces nn.Conv2d(64, n, 3, padding=1) forward / input-gradient of the reference
// (sres/model/common/cnn.py:8-9 used at sres/model/rcan/network.py:14-16,55,71, blocks.py:62-64).
#include "ptx.cuh"
#include "internal.h"
#include "conv_epi.cuh"

namespace sres {

constexpr int kMaxStages = 6;
constexpr int kBoxRows = 64;   // rows per TMA box of the A operand (8 KB)
constexpr int kAccStages = 4;  // TMEM accumulator ring
constexpr int kConvThreads = 384;

struct ConvKParams {
  int B, H, W, P, R;      // input geometry, P = W+1, R = H+1
  int npos;               // rows of the input PTL
  int n_tiles;            // 128-row tiles
  int nstage;             // smem ring depth
  int stage_rows;         // rows per smem ring slot (multiple of box_rows)
  int box_rows;           // rows per TMA box of the A operand: the whole halo window when it fits one box (<= 256 rows)
  int n_out, c_real;
  unsigned flags;
  int map_mode, sub_i, sub_j, sf;
  const float* bias;
  const float* resid;
  const float* resid2;
  const uint16_t* mask;
  float* out_f32;
  uint16_t* out_bf16;
  float* pool_part;
  float* out_nchw;
  // TMA-staged epilogue (identity mapping): per-warp slabs in shared memory
  int tma_epi;          // 1: outputs / addends go through smem slabs + TMA, 0: direct global accesses
  int use_o16, use_msk, use_r32, use_o32;
  int off_s16, off_msk, off_s32, off_tail;  // byte offsets from the aligned smem base
  long long* timeline;  // bring-up only: per-CTA clock stamps [grid][16]
};

// FL >= 0: an instance specialised at compile time for one epilogue flavour of the TMA-staged path (bit set below);
// the RCAB loop's four convolutions each get one, which keeps the epilogue's code and instruction count small --
// it shares the SM's issue ports and instruction cache with the single MMA-issuing thread.  The specialised pooled /
// dot-product instances reduce their columns in the fragment layout; FL = -1 is the generic kernel (runtime flags, all
// mappings, column sums in the row layout).
constexpr int kFlO16 = 1, kFlO32 = 2, kFlR32 = 4, kFlMsk = 8, kFlRelu = 16, kFlPool = 32, kFlDot = 64;
template <int N_OUT, int FL>
__global__ void __launch_bounds__(kConvThreads, 1)
conv3x3_igemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW,
                     const __grid_constant__ CUtensorMap tmO16, const __grid_constant__ CUtensorMap tmMsk,
                     const __grid_constant__ CUtensorMap tmR32, const __grid_constant__ CUtensorMap tmO32,
                     const ConvKParams p) {
  extern __shared__ uint8_t smem_raw[];
  // 1024-B aligned carve-up (128B swizzle atoms are 1024 B).
  // offset arithmetic (not an integer round trip) keeps the pointer in the shared address space: LDS/STS, not generic LD/ST
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  constexpr int kWBytes = 9 * N_OUT * 128;
  uint8_t* smem_w = smem;
  uint8_t* smem_a = smem + kWBytes;
  const int stage_bytes = p.stage_rows * 128;
  uint8_t* tail = smem + p.off_tail;
  uint64_t* bar_full = reinterpret_cast<uint64_t*>(tail);  // [kMaxStages]
  uint64_t* bar_empty = bar_full + kMaxStages;              // [kMaxStages]
  uint64_t* bar_w = bar_empty + kMaxStages;                 // [1]
  uint64_t* bar_tfull = bar_w + 1;                          // [kAccStages]
  uint64_t* bar_tempty = bar_tfull + kAccStages;            // [kAccStages]
  uint64_t* bar_in = bar_tempty + kAccStages;               // [8] epilogue operand loads, one per warp
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(bar_in + 8);
  float* s_bias = reinterpret_cast<float*>(tmem_holder + 2);  // [N_OUT]

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);  // warp-uniform by construction
  const int lane = threadIdx.x & 31;
  long long* tl = p.timeline ? p.timeline + (size_t)blockIdx.x * 16 : nullptr;
#define SRES_STAMP(i)                                   \
  do {                                                  \
    if (tl && lane == 0) tl[i] = clock64();             \
  } while (0)
  if (tl && threadIdx.x == 0) {
    unsigned long long gt;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt));
    tl[10] = (long long)gt;
    tl[0] = clock64();
    tl[13] = tl[14] = tl[15] = 0;
  }
  constexpr uint32_t tmem_cols = (kAccStages * N_OUT) < 32 ? 32 : (kAccStages * N_OUT);

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmW);
    for (int i = 0; i < kMaxStages; ++i) {
      mbar_init(&bar_full[i], 1);
      mbar_init(&bar_empty[i], 1);
    }
    mbar_init(bar_w, 1);
    for (int i = 0; i < kAccStages; ++i) {
      mbar_init(&bar_tfull[i], 1);
      mbar_init(&bar_tempty[i], 8);  // one arrive per epilogue warp
    }
    for (int i = 0; i < 8; ++i) mbar_init(&bar_in[i], 1);
    mbar_fence_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_holder, tmem_cols);
    tmem_relinquish();
  }
  if (threadIdx.x < N_OUT) s_bias[threadIdx.x] = p.bias ? p.bias[threadIdx.x] : 0.f;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_holder, 0);
  if (warp == 0) SRES_STAMP(1);
  pdl_launch_dependents();  // the next kernel may start its prologue as soon as SMs free up

  if (warp == 0) {
    // ===================== TMA producer (whole warp runs the loop, one elected lane issues) ==========
    const bool leader = elect_one();
    if (leader) {
      mbar_expect_tx(bar_w, kWBytes);
      for (int t = 0; t < 9; ++t) tma_load_2d(smem_w + t * N_OUT * 128, &tmW, bar_w, 0, t * N_OUT);
    }
    pdl_wait();  // the packed weights are old; the activations come from the previous kernel
    int it = 0;
    for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++it) {
      const int slot = it % p.nstage;
      const uint32_t ph = (it / p.nstage) & 1;
      mbar_wait(&bar_empty[slot], ph ^ 1, 1);
      const int row0 = tile * 128 - (p.P + 1);
      uint8_t* dst = smem_a + slot * stage_bytes;
      if (leader) {
        mbar_expect_tx(&bar_full[slot], stage_bytes);
        for (int r = 0; r < p.stage_rows; r += p.box_rows) tma_load_2d(dst + r * 128, &tmA, &bar_full[slot], 0, row0 + r);
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (whole warp runs the loop, one elected lane issues) ==========
    const bool leader = elect_one();
    constexpr uint32_t idesc = make_idesc_bf16(128, N_OUT, 0, 0);
    constexpr uint32_t dhi = sdesc_hi_sw128(1024);
    const uint32_t w_lo = sdesc_lo(smem_u32(smem_w), 16);
    const uint32_t a_lo0 = sdesc_lo(smem_u32(smem_a), 16);
    const uint32_t row_step = uint32_t(p.P) * 8;  // one image row of the halo window, in 16-byte units
    mbar_wait(bar_w, 0, 2);
    SRES_STAMP(3);
    int it = 0;
    for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++it) {
      const int slot = it % p.nstage;
      const uint32_t ph = (it / p.nstage) & 1;
      const int acc = it % kAccStages;
      const uint32_t aph = (it / kAccStages) & 1;
      long long w0 = 0, w1 = 0;
      if (tl) w0 = clock64();
      mbar_wait(&bar_tempty[acc], aph ^ 1, 3);
      if (tl) w1 = clock64();
      mbar_wait(&bar_full[slot], ph, 4);
      if (tl && lane == 0) { tl[14] += w1 - w0; tl[15] += clock64() - w1; }   // waiting for the epilogue / for TMA
      if (it == 0) SRES_STAMP(4);
      tc_fence_after();
      const uint32_t a_tile = a_lo0 + uint32_t(slot * stage_bytes) / 16;
      const uint32_t d_tmem = tmem_base + uint32_t(acc * N_OUT);
      if (leader) {
#pragma unroll
        for (int t = 0; t < 9; ++t) {
          const uint32_t a_tap = a_tile + uint32_t(t / 3) * row_step + uint32_t(t % 3) * 8;
          const uint32_t b_tap = w_lo + uint32_t(t * N_OUT * 8);
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            if (t == 0 && k == 0) umma_bf16_lohi<false>(d_tmem, a_tap, dhi, b_tap, dhi, idesc);
            else umma_bf16_lohi<true>(d_tmem, a_tap + k * 2, dhi, b_tap + k * 2, dhi, idesc);
          }
        }
        umma_commit(&bar_empty[slot]);  // smem slot free once these MMAs retire
        umma_commit(&bar_tfull[acc]);   // accumulator ready
      }
      __syncwarp();
    }
    SRES_STAMP(5);
  } else if (warp >= 4) {
    // ===================== epilogue =====================
    const int ew = warp - 4;        // 0..7
    const int wq = warp & 3;        // TMEM lane quarter this warp may access
    const int half = ew >> 2;       // which 32 of the 64 output columns
    constexpr int NCH = (N_OUT == 64) ? 2 : 1;          // 16-column chunks this warp handles
    const bool has_work = (N_OUT == 64) || half == 0;   // narrow conv: 16 columns, first half only
    const int RP = p.R * p.P;
    uint8_t* s16 = smem + p.off_s16 + ew * 2048;   // 32 rows x 64 B (bf16, 64B swizzle)
    uint8_t* smk = smem + p.off_msk + ew * 2048;
    uint8_t* s32 = smem + p.off_s32 + ew * 4096;   // 32 rows x 128 B (fp32 half rows, 128B swizzle)
    uint64_t* bin = &bar_in[ew];
    constexpr bool kSpec = FL >= 0;
    constexpr bool FRAG = kSpec && (FL & (kFlPool | kFlDot));
    const bool f_tma = kSpec ? true : bool(p.tma_epi);
    const bool f_o16 = kSpec ? bool(FL & kFlO16) : bool(p.use_o16);
    const bool f_o32 = kSpec ? bool(FL & kFlO32) : bool(p.use_o32);
    const bool f_r32 = kSpec ? bool(FL & kFlR32) : bool(p.use_r32);
    const bool f_msk = kSpec ? bool(FL & kFlMsk) : bool(p.use_msk);
    const bool f_relu = kSpec ? bool(FL & kFlRelu) : bool(p.flags & SRES_EPI_RELU);
    const bool f_pool = kSpec ? bool(FL & kFlPool) : bool(p.flags & SRES_EPI_POOL);
    const bool f_dot = kSpec ? bool(FL & kFlDot) : bool(p.flags & SRES_EPI_DOT);
    const float* f_res2 = kSpec ? nullptr : p.resid2;
    const bool use_in = f_tma && (f_msk | f_r32);
    // per-tile column reductions (pooled sums / channel-attention dot products) run in the fragment layout
    const int fm = lane & 3, frq = lane >> 2;            // fragment column pair / row within an 8-row group
    const int fcol = ((lane >> 4) & 1) * 16 + ((lane >> 3) & 1) * 8 + 2 * fm + ((lane >> 2) & 1);  // column after frag_colsum
    float bias8[8];
    if constexpr (FRAG) {
#pragma unroll
      for (int i = 0; i < 8; ++i) bias8[i] = s_bias[(half * 32 + 8 * (i >> 1) + 2 * fm + (i & 1)) % N_OUT];
    }
    pdl_wait();
    int it = 0;
    for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++it) {
      const int acc = it % kAccStages;
      const uint32_t aph = (it / kAccStages) & 1;
      const int row0 = tile * 128 + wq * 32;
      if (f_tma) {
        // the slab must have been read out by the previous tile's TMA stores; then prefetch this tile's
        // fp32 addend / mask while the tensor core is still working on it
        if (lane == 0) {
          bulk_wait_read<0>();
          if (use_in) {
            mbar_expect_tx(bin, (f_msk ? 2048u : 0u) + (f_r32 ? 4096u : 0u));
            if (f_msk) tma_load_2d(smk, &tmMsk, bin, half * 32, row0);
            if (f_r32) tma_load_2d(s32, &tmR32, bin, half * 32, row0);
          }
        }
        __syncwarp();
      }
      long long e0 = 0;
      if (tl && warp == 4) e0 = clock64();
      mbar_wait(&bar_tfull[acc], aph, 5);
      if (tl && warp == 4 && lane == 0) tl[13] += clock64() - e0;   // epilogue idle, waiting for the tensor core
      if (warp == 4) { if (it == 0) SRES_STAMP(6); SRES_STAMP(7); }
      tc_fence_after();
      if (has_work) {
        const int q = row0 + lane;
        const bool inrange = q < p.npos;
        const int b = q / RP;
        const int rem = q - b * RP;
        const int y = rem / p.P;
        const int x = rem - y * p.P;
        const bool pad = (x == p.W) || (y == p.H) || !inrange;
        const int seg = (b != (tile * 128) / RP) ? 1 : 0;
        const uint32_t trow = tmem_base + (uint32_t(wq * 32) << 16) + uint32_t(acc * N_OUT + half * 32);
        if constexpr (FRAG) {
          // ---------------- fragment-layout epilogue: thread = rows frq + 8j (j < 4) x column pairs 8k + 2fm ----------------
          uint32_t fa[16], fb[16];
          tmem_ld_frag16(trow, fa);
          tmem_ld_frag16(trow + (16u << 16), fb);
          const unsigned padmask = __ballot_sync(0xffffffffu, pad);
          const unsigned seg1 = __ballot_sync(0xffffffffu, seg == 1);
          const bool mixed = seg1 != 0u && seg1 != 0xffffffffu;   // the warp's rows straddle two images
          tmem_ld_wait();
          if (use_in) mbar_wait(bin, it & 1, 6);
          const int sw3 = (frq >> 1) & 3;
          float cs0[8], cs1[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) cs0[i] = cs1[i] = 0.f;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int r = frq + 8 * j;
            const bool rpad = (padmask >> r) & 1u;
            const bool rs1 = (seg1 >> r) & 1u;
            uint8_t* row32 = s32 + r * 128 + (fm & 1) * 8;
            uint8_t* row16 = s16 + r * 64 + 4 * fm;
            const uint8_t* rowmk = smk + r * 64 + 4 * fm;
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
              if (f_relu) { v0 = fmaxf(v0, 0.f); v1 = fmaxf(v1, 0.f); }
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
          // one column total per lane; an unmixed warp belongs to exactly one image segment
          const float t0 = frag_colsum(cs0, lane);
          const float t1 = mixed ? frag_colsum(cs1, lane) : 0.f;
          float* dst = p.pool_part + ((long long)tile * 2 * 4 + wq) * 64 + half * 32 + fcol;
          const bool all1 = seg1 == 0xffffffffu;
          dst[0] = all1 ? 0.f : t0;
          dst[4 * 64] = all1 ? t0 : t1;
        } else {
        uint32_t raw[16 * NCH];
        if constexpr (N_OUT == 64) {
          tmem_ld32(trow, raw);
        } else {
          tmem_ld16(trow, raw);
        }
        tmem_ld_wait();
        if (f_tma) {
          // ---------------- TMA-staged epilogue (identity mapping, 64 outputs) ----------------
          if (use_in) mbar_wait(bin, it & 1, 6);
          const int sw7 = lane & 7, sw3 = (lane >> 1) & 3;
          uint8_t* r16 = s16 + lane * 64;
          const uint8_t* rmk = smk + lane * 64;
          uint8_t* r32 = s32 + lane * 128;
#pragma unroll
          for (int ch = 0; ch < NCH; ++ch) {
            const int c0 = half * 32 + ch * 16;  // first output column of this chunk
            float v[16];
#pragma unroll
            for (int j = 0; j < 4; ++j) {   // 128-bit broadcast loads: shared-memory instructions are the scarce resource here
              const float4 b4 = *reinterpret_cast<const float4*>(s_bias + c0 + 4 * j);
              v[4 * j + 0] = __uint_as_float(raw[ch * 16 + 4 * j + 0]) + b4.x;
              v[4 * j + 1] = __uint_as_float(raw[ch * 16 + 4 * j + 1]) + b4.y;
              v[4 * j + 2] = __uint_as_float(raw[ch * 16 + 4 * j + 2]) + b4.z;
              v[4 * j + 3] = __uint_as_float(raw[ch * 16 + 4 * j + 3]) + b4.w;
            }
            if (f_r32) {
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const float4 r = *reinterpret_cast<const float4*>(r32 + (((ch * 4 + j) ^ sw7) << 4));
                v[4 * j + 0] += r.x; v[4 * j + 1] += r.y; v[4 * j + 2] += r.z; v[4 * j + 3] += r.w;
              }
            }
            if (f_res2 && inrange) {
              const float4* rp = reinterpret_cast<const float4*>(f_res2 + (long long)q * 64 + c0);
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const float4 r = rp[j];
                v[4 * j + 0] += r.x; v[4 * j + 1] += r.y; v[4 * j + 2] += r.z; v[4 * j + 3] += r.w;
              }
            }
            if (f_relu) {
#pragma unroll
              for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.f);
            }
            if (f_msk && !f_dot) {
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
            if (f_dot) {
              // per-image channel sums of v * other (the channel-attention backward reduction, fused here)
              float t[16];
#pragma unroll
              for (int j = 0; j < 2; ++j) {
                const uint4 mk = *reinterpret_cast<const uint4*>(rmk + (((ch * 2 + j) ^ sw3) << 4));
                const uint32_t w4[4] = {mk.x, mk.y, mk.z, mk.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  t[8 * j + 2 * e] = v[8 * j + 2 * e] * bf16_lo(w4[e]);
                  t[8 * j + 2 * e + 1] = v[8 * j + 2 * e + 1] * bf16_hi(w4[e]);
                }
              }
              pool_partials(t, seg, lane, p.pool_part + ((long long)tile * 2 * 4 + wq) * 64 + c0);
            }
            if (f_o32) {
#pragma unroll
              for (int j = 0; j < 4; ++j)
                *reinterpret_cast<float4*>(r32 + (((ch * 4 + j) ^ sw7) << 4)) =
                    make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
            }
            if (f_o16) {
#pragma unroll
              for (int j = 0; j < 2; ++j)
                *reinterpret_cast<uint4*>(r16 + (((ch * 2 + j) ^ sw3) << 4)) =
                    make_uint4(pack_bf16x2(v[8 * j], v[8 * j + 1]), pack_bf16x2(v[8 * j + 2], v[8 * j + 3]),
                               pack_bf16x2(v[8 * j + 4], v[8 * j + 5]), pack_bf16x2(v[8 * j + 6], v[8 * j + 7]));
            }
            if (f_pool) pool_partials(v, seg, lane, p.pool_part + ((long long)tile * 2 * 4 + wq) * 64 + c0);
          }
        } else {
          // ---------------- direct epilogue (PixelShuffle scatter / planar output / narrow conv) ----------------
          long long oq = q;
          bool ovalid = inrange;
          if (p.map_mode == SRES_MAP_SHUFFLE) {
            const int P2 = p.sf * p.W + 1, R2 = p.sf * p.H + 1;
            const int oy = p.sf * y + p.sub_i, ox = p.sf * x + p.sub_j;
            ovalid = inrange && oy < R2 && ox < P2;
            oq = (long long)b * R2 * P2 + (long long)oy * P2 + ox;
          } else if (p.map_mode == SRES_MAP_UNSHUFFLE) {
            const int Pl = p.W / p.sf + 1, Rl = p.H / p.sf + 1;
            const int sub = (y % p.sf) * p.sf + (x % p.sf);
            oq = (long long)sub * p.B * Rl * Pl + (long long)b * Rl * Pl + (long long)(y / p.sf) * Pl + (x / p.sf);
          }
#pragma unroll
          for (int ch = 0; ch < NCH; ++ch) {
            const int c0 = half * 32 + ch * 16;
            float v[16];
#pragma unroll
            for (int j = 0; j < 4; ++j) {   // 128-bit broadcast loads: shared-memory instructions are the scarce resource here
              const float4 b4 = *reinterpret_cast<const float4*>(s_bias + c0 + 4 * j);
              v[4 * j + 0] = __uint_as_float(raw[ch * 16 + 4 * j + 0]) + b4.x;
              v[4 * j + 1] = __uint_as_float(raw[ch * 16 + 4 * j + 1]) + b4.y;
              v[4 * j + 2] = __uint_as_float(raw[ch * 16 + 4 * j + 2]) + b4.z;
              v[4 * j + 3] = __uint_as_float(raw[ch * 16 + 4 * j + 3]) + b4.w;
            }
            if (p.resid && ovalid) {
              const float4* rp = reinterpret_cast<const float4*>(p.resid + oq * 64 + c0);
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const float4 r = rp[j];
                v[4 * j + 0] += r.x; v[4 * j + 1] += r.y; v[4 * j + 2] += r.z; v[4 * j + 3] += r.w;
              }
            }
            if (f_res2 && ovalid) {
              const float4* rp = reinterpret_cast<const float4*>(f_res2 + oq * 64 + c0);
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const float4 r = rp[j];
                v[4 * j + 0] += r.x; v[4 * j + 1] += r.y; v[4 * j + 2] += r.z; v[4 * j + 3] += r.w;
              }
            }
            if (f_relu) {
#pragma unroll
              for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.f);
            }
            if (p.mask && inrange) {
              const uint4* mp = reinterpret_cast<const uint4*>(p.mask + (long long)q * 64 + c0);
#pragma unroll
              for (int j = 0; j < 2; ++j) {
                const uint4 mk = mp[j];
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
            if (ovalid) {
              if (p.out_f32) {
                float4* op = reinterpret_cast<float4*>(p.out_f32 + oq * 64 + c0);
#pragma unroll
                for (int j = 0; j < 4; ++j) op[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
              }
              if (p.out_bf16) {
                uint4* op = reinterpret_cast<uint4*>(p.out_bf16 + oq * 64 + c0);
#pragma unroll
                for (int j = 0; j < 2; ++j)
                  op[j] = make_uint4(pack_bf16x2(v[8 * j], v[8 * j + 1]), pack_bf16x2(v[8 * j + 2], v[8 * j + 3]),
                                     pack_bf16x2(v[8 * j + 4], v[8 * j + 5]), pack_bf16x2(v[8 * j + 6], v[8 * j + 7]));
              }
              if (p.out_nchw && !pad) {
#pragma unroll
                for (int c = 0; c < 16; ++c)   // unrolled + predicated: v[] stays in registers
                  if (c0 + c < p.c_real) p.out_nchw[(((long long)b * p.c_real + c0 + c) * p.H + y) * p.W + x] = v[c];
              }
            }
            if (f_pool) pool_partials(v, seg, lane, p.pool_part + ((long long)tile * 2 * 4 + wq) * 64 + c0);
          }
        }
        }
      }
      // accumulator stage drained (all tcgen05.ld of this warp have completed)
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_tempty[acc]);
      if (f_tma) {
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          if (f_o16) tma_store_2d(&tmO16, s16, half * 32, row0);
          if (f_o32) tma_store_2d(&tmO32, s32, half * 32, row0);
          bulk_commit();
        }
      }
    }
    if (warp == 4) SRES_STAMP(8);
    if ((FL >= 0 || p.tma_epi) && lane == 0) bulk_wait_all<0>();
    if (warp == 4) SRES_STAMP(9);
  }

  tc_fence_before();
  __syncthreads();
  if (tl && threadIdx.x == 0) {
    unsigned long long gt;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt));
    tl[11] = (long long)gt;
    tl[12] = clock64();
  }
  if (warp == 2) tmem_dealloc(tmem_base, tmem_cols);
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
static int launch_conv(const sres_conv_args* a, cudaStream_t stream) {
  if (!a || !a->in_bf16 || !a->wpack_bf16) return set_error(SRES_ERR_INVALID_ARG, "conv: null input");
  if (a->n_out != 64 && a->n_out != 16) return set_error(SRES_ERR_UNSUPPORTED, "conv: n_out must be 64 or 16");
  if (a->B <= 0 || a->H <= 0 || a->W <= 0) return set_error(SRES_ERR_INVALID_ARG, "conv: bad geometry");
  const int sf = a->shuffle_factor > 0 ? a->shuffle_factor : 2;
  if (a->map_mode == SRES_MAP_UNSHUFFLE && (a->H % sf || a->W % sf))
    return set_error(SRES_ERR_INVALID_ARG, "conv: unshuffle factor must divide H and W");
  if ((a->epi_flags & (SRES_EPI_POOL | SRES_EPI_DOT)) && !a->pool_part) return set_error(SRES_ERR_INVALID_ARG, "conv: pool_part missing");
  if ((a->epi_flags & SRES_EPI_DOT) && ((a->epi_flags & SRES_EPI_POOL) || !a->mask_bf16 || a->map_mode != SRES_MAP_IDENT || a->n_out != 64 ||
                                         a->out_nchw || (a->debug_flags & 2)))
    return set_error(SRES_ERR_INVALID_ARG, "conv: SRES_EPI_DOT needs mask_bf16 (the other factor), identity mapping, 64 outputs and no SRES_EPI_POOL");

  // tail convolution (16 packed output rows, planar output): the three-taps-per-MMA kernel of conv_n192.cu, whose halo
  // staging does not grow with the image width (debug_flags bits 1 and 6 keep the tap-per-MMA kernel)
  if (a->n_out == 16 && a->out_nchw && a->map_mode == SRES_MAP_IDENT && !a->out_f32 && !a->out_bf16 && !a->resid_f32 &&
      !a->resid2_f32 && !a->mask_bf16 && !(a->epi_flags & (SRES_EPI_POOL | SRES_EPI_DOT)) && a->c_real >= 1 && a->c_real <= 16 &&
      !(a->debug_flags & (2 | 64)) && conv_n48_available(a->H, a->W))
    return launch_conv_n48(a, stream);
  ConvKParams p{};
  p.B = a->B; p.H = a->H; p.W = a->W; p.P = a->W + 1; p.R = a->H + 1;
  const long long npos = (long long)p.B * p.R * p.P;
  if (npos > 0x7fffff00LL) return set_error(SRES_ERR_UNSUPPORTED, "conv: batch too large for 32-bit rows");
  p.npos = (int)npos;
  p.n_tiles = (p.npos + 127) / 128;
  p.n_out = a->n_out; p.c_real = a->c_real;
  p.flags = a->epi_flags; p.map_mode = a->map_mode; p.sub_i = a->sub_i; p.sub_j = a->sub_j; p.sf = sf;
  p.bias = a->bias; p.resid = a->resid_f32; p.resid2 = a->resid2_f32; p.mask = (const uint16_t*)a->mask_bf16;
  p.out_f32 = a->out_f32; p.out_bf16 = (uint16_t*)a->out_bf16; p.pool_part = a->pool_part; p.out_nchw = a->out_nchw;
  p.timeline = (long long*)a->debug_timeline;
  // TMA-staged epilogue whenever rows map to themselves; scattered (PixelShuffle) and planar stores go direct
  p.tma_epi = (a->map_mode == SRES_MAP_IDENT && a->n_out == 64 && !a->out_nchw && !(a->debug_flags & 2)) ? 1 : 0;
  if (p.tma_epi) {
    p.use_o16 = a->out_bf16 != nullptr; p.use_msk = a->mask_bf16 != nullptr;
    p.use_r32 = a->resid_f32 != nullptr; p.use_o32 = a->out_f32 != nullptr;
  }
  const int wbytes = 9 * a->n_out * 128;
  const int smem_max = 232448;  // 227 KB
  const int tail_bytes = 1024;
  int slab_bytes = (p.use_o16 ? 16384 : 0) + (p.use_msk ? 16384 : 0) + ((p.use_r32 | p.use_o32) ? 32768 : 0);
  const int rows = 128 + 2 * (p.P + 1);
  // one TMA box of the exact window (rounded to the 8-row swizzle atom) when it fits the 256-row box limit: fewer bytes
  // into shared memory (232 instead of 256 rows at 48x48) and one TMA instruction per tile instead of four
  const bool one_box = (rows + 7) / 8 * 8 <= 256;
  p.box_rows = one_box ? (rows + 7) / 8 * 8 : kBoxRows;
  p.stage_rows = (rows + p.box_rows - 1) / p.box_rows * p.box_rows;
  int ns = (smem_max - 1024 - wbytes - tail_bytes - slab_bytes) / (p.stage_rows * 128);
  if (ns < 1 && p.tma_epi && !(a->epi_flags & SRES_EPI_DOT)) {  // wide image: give the slab space to the halo window
    p.tma_epi = p.use_o16 = p.use_msk = p.use_r32 = p.use_o32 = 0;
    slab_bytes = 0;
    ns = (smem_max - 1024 - wbytes - tail_bytes) / (p.stage_rows * 128);
  }
  if (ns > kMaxStages) ns = kMaxStages;
  if (ns < 1) return set_error(SRES_ERR_UNSUPPORTED, "conv: image too wide for the flat halo window");
  p.nstage = ns;
  int off = wbytes + p.nstage * p.stage_rows * 128;
  p.off_s16 = off; off += p.use_o16 ? 16384 : 0;
  p.off_msk = off; off += p.use_msk ? 16384 : 0;
  p.off_s32 = off; off += (p.use_r32 | p.use_o32) ? 32768 : 0;
  p.off_tail = off; off += tail_bytes;
  const size_t smem = (size_t)off + 1024;  // + alignment slack

  CUtensorMap tmA, tmW, tmO16, tmMsk, tmR32, tmO32;
  int rc = make_tmap_rows64(&tmA, a->in_bf16, (uint64_t)p.npos, p.box_rows);
  if (rc) return rc;
  rc = make_tmap_rows64(&tmW, a->wpack_bf16, (uint64_t)(9 * a->n_out), a->n_out);
  if (rc) return rc;
  tmO16 = tmA; tmMsk = tmA; tmR32 = tmA; tmO32 = tmA;
  if (p.tma_epi) {
    if (p.use_o16 && (rc = make_tmap_rows64_half(&tmO16, a->out_bf16, (uint64_t)p.npos, 32))) return rc;
    if (p.use_msk && (rc = make_tmap_rows64_half(&tmMsk, a->mask_bf16, (uint64_t)p.npos, 32))) return rc;
    if (p.use_r32 && (rc = make_tmap_rows64_f32(&tmR32, a->resid_f32, (uint64_t)p.npos, 32))) return rc;
    if (p.use_o32 && (rc = make_tmap_rows64_f32(&tmO32, a->out_f32, (uint64_t)p.npos, 32))) return rc;
  }

  int sms = device_sm_count();
  if (sms <= 0) return set_error(SRES_ERR_NO_DEVICE, "conv: no CUDA device");
  const int grid = persistent_grid(p.n_tiles, sms);
  cudaError_t e = cudaSuccess;
  int dev = 0;
  cudaGetDevice(&dev);
  // compile-time flavour of the TMA-staged epilogue, if this call is one of the specialised ones
  int fl = -1;
  if (p.tma_epi && !a->resid2_f32 && !(a->debug_flags & 16)) {
    fl = (p.use_o16 ? kFlO16 : 0) | (p.use_o32 ? kFlO32 : 0) | (p.use_r32 ? kFlR32 : 0) | (p.use_msk ? kFlMsk : 0) |
         ((a->epi_flags & SRES_EPI_RELU) ? kFlRelu : 0) | ((a->epi_flags & SRES_EPI_POOL) ? kFlPool : 0) |
         ((a->epi_flags & SRES_EPI_DOT) ? kFlDot : 0);
  }
#define SRES_CONV_CASE(NOUT, FLV)                                                                                        \
  {                                                                                                                      \
    static thread_local int attr_dev = -1;                                                                               \
    if (attr_dev != dev) {                                                                                               \
      e = cudaFuncSetAttribute(conv3x3_igemm_kernel<NOUT, FLV>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);  \
      if (e != cudaSuccess) return set_cuda_error(e, "conv: smem attribute");                                           \
      attr_dev = dev;                                                                                                    \
    }                                                                                                                    \
    e = launch_pdl(conv3x3_igemm_kernel<NOUT, FLV>, dim3(grid), dim3(kConvThreads), smem, stream, tmA, tmW, tmO16, tmMsk, \
                   tmR32, tmO32, p);                                                                                     \
  }
  if (a->n_out == 16) {
    SRES_CONV_CASE(16, -1)
  } else {
    switch (fl) {
      case kFlRelu | kFlO16: SRES_CONV_CASE(64, kFlRelu | kFlO16) break;                                  // RCAB conv1
      case kFlPool | kFlO16: SRES_CONV_CASE(64, kFlPool | kFlO16) break;                                  // RCAB conv2
      case kFlMsk | kFlO16: SRES_CONV_CASE(64, kFlMsk | kFlO16) break;                                    // dgrad of conv2
      case kFlR32 | kFlO32 | kFlMsk | kFlDot: SRES_CONV_CASE(64, kFlR32 | kFlO32 | kFlMsk | kFlDot) break;    // dgrad of conv1
      case kFlR32 | kFlO32 | kFlO16: SRES_CONV_CASE(64, kFlR32 | kFlO32 | kFlO16) break;                  // EDSR conv2 / conv1 dgrad
      case kFlO32 | kFlMsk | kFlDot: SRES_CONV_CASE(64, kFlO32 | kFlMsk | kFlDot) break;                  // dgrad of a group tail
      default: SRES_CONV_CASE(64, -1) break;
    }
  }
#undef SRES_CONV_CASE
  if (e != cudaSuccess) return set_cuda_error(e, "conv: launch");
  e = cudaGetLastError();
  if (e != cudaSuccess) return set_cuda_error(e, "conv: launch");
  return SRES_OK;
}

}  // namespace sres

extern "C" int sres_conv_tile_rows(int H, int W) {
  (void)H; (void)W;
  return 128;
}

extern "C" int sres_conv_mtiles(int B, int H, int W) {
  const long long npos = (long long)B * (H + 1) * (W + 1);
  const int tr = sres_conv_tile_rows(H, W);
  return (int)((npos + tr - 1) / tr);
}

extern "C" int sres_conv_supported(int H, int W, int n_out) {
  if (n_out == 16 && sres::conv_n48_available(H, W)) return 1;
  const int wbytes = 9 * n_out * 128;
  const int rows = 128 + 2 * (W + 2);
  const int stage_rows = (rows + sres::kBoxRows - 1) / sres::kBoxRows * sres::kBoxRows;
  // one ring slot next to the weights (the epilogue falls back to direct stores when its slabs do not fit)
  return (232448 - 1024 - wbytes - 1024) / (stage_rows * 128) >= 1 ? 1 : 0;
}

extern "C" int sres_conv3x3_igemm(const sres_conv_args* args, void* stream) {
  return sres::launch_conv(args, (cudaStream_t)stream);
}
