// Tail convolution 64 -> Cout <= 16 over the padded tile layout with the three horizontal taps stacked on the UMMA N
// dimension (sm_100a), planar fp32 output.
//
// The weights are packed with 16 output rows per tap.  One instruction covers the three taps (ky, 0..2) of a kernel row:
//
//     D_kx[i] = sum_ky  X[m_i + (ky-1) P] . W(ky, kx)          N = 48 = 3 x 16 output features, 12 MMAs per tile
//     out[m_i] = D_0[i-1] + D_1[i] + D_2[i+1]                   (P = W+1: one image row of the padded tile layout)
//
// B for kernel row ky is simply taps 3ky..3ky+2 of the packed weights, which are contiguous (48 rows).  The three
// 16-column accumulators of a tile are added with a shift of one TMEM lane (= one PTL row) in the epilogue.  A warp owns
// 32 lanes, so the shift is a lane rotation by warp shuffle; the two rows that cross a warp's lane quarter travel
// through a small shared-memory exchange, and because the first and last MMA row of a tile have no neighbour the tiles
// overlap by two rows: a tile is 128 MMA rows = 126 output rows.
//
// The A operand of kernel row ky is the 128-row block starting (ky-1) P rows from the tile, so the halo window is
// 128 + 2P rows (one TMA box when it fits 256 rows), or -- for wide images, where that window would not fit --
// three independent 128-row boxes: the shared-memory footprint does not grow with the image width (x8 upscaling
// of 96 x 96 tiles, BASELINE config 5's 768-pixel rows).
//
// (The 64 -> 64 form of this kernel, N = 192, lost to the tap-per-MMA kernel of conv_igemm.cu and was removed: DESIGN.md
// section 3.1a.)
//
// Replaces nn.Conv2d(64, Cout, 3, padding=1) forward of the reference's tail conv (sres/model/rcan/network.py:16).
#include "ptx.cuh"
#include "internal.h"

namespace sres {

constexpr int kNStages = 6;
constexpr int kNWarps = 18;             // 0 = TMA producer (+ TMEM allocation), 1 = MMA issuer, 2..17 = two epilogue groups
constexpr int kNThreads = kNWarps * 32;
constexpr int kNTileOut = 126;          // output rows per tile (128 MMA rows, one halo row on each side)
constexpr int kNB = 16;                 // output features per horizontal tap
constexpr int kNWBytes = 9 * kNB * 128; // packed weights, all taps

struct ConvN48Params {
  int H, W, P, R;
  int npos, n_tiles;
  int nstage, stage_bytes;
  int nbox, box_rows;  // TMA boxes per ring slot and their height
  int box_step;        // PTL rows between consecutive boxes: box_rows (split union window) or P (one block per kernel row)
  int ky_step16;       // distance between the A blocks of consecutive kernel rows, in 16-byte units
  unsigned flags;
  const float* bias;
  float* out_nchw;     // planar fp32 output (B, c_real, H, W)
  int c_real;
  int off_xch, off_tail;
  long long* timeline;
};

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// Warp roles (576 threads): 0 = TMA producer, 1 = MMA issuer, 2..9 = epilogue group 0, 10..17 = epilogue group 1.
// Group g drains accumulator stage g, i.e. every second tile of the CTA; in each group one warp per TMEM lane quarter
// has work.
__global__ void __launch_bounds__(kNThreads, 1)
conv3x3_n48_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW,
                   const __grid_constant__ ConvN48Params p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);  // offset arithmetic keeps LDS/STS
  uint8_t* smem_w = smem;
  constexpr int kWRow = 3 * kNB * 128;  // bytes of one kernel row of the packed weights (three taps)
  uint8_t* smem_a = smem + 3 * kWRow;
  uint8_t* tail = smem + p.off_tail;
  uint64_t* bar_full = reinterpret_cast<uint64_t*>(tail);  // [kNStages]
  uint64_t* bar_empty = bar_full + kNStages;                // [kNStages]
  uint64_t* bar_w = bar_empty + kNStages;                   // [3] one per kernel row of the weights
  uint64_t* bar_tfull = bar_w + 3;                          // [2]
  uint64_t* bar_tempty = bar_tfull + 2;                     // [2]
  uint64_t* bar_in = bar_tempty + 2;                        // [16]
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(bar_in + 16);
  float* s_bias = reinterpret_cast<float*>(tmem_holder + 2);  // [64]

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  long long* tl = p.timeline ? p.timeline + (size_t)blockIdx.x * 16 : nullptr;
#define N48_STAMP(i)                           \
  do {                                         \
    if (tl && lane == 0) tl[i] = clock64();    \
  } while (0)
  if (tl && threadIdx.x == 0) {
    tl[0] = clock64();
    tl[13] = tl[14] = tl[15] = 0;
  }

  if (threadIdx.x == 32) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmW);
    for (int i = 0; i < kNStages; ++i) {
      mbar_init(&bar_full[i], 1);
      mbar_init(&bar_empty[i], 1);
    }
    for (int i = 0; i < 3; ++i) mbar_init(&bar_w[i], 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&bar_tfull[i], 1);
      mbar_init(&bar_tempty[i], 4);  // one arrive per warp of the group that drains the stage
    }
    for (int i = 0; i < 16; ++i) mbar_init(&bar_in[i], 1);
    mbar_fence_init();
  }
  if (warp == 0) {
    tmem_alloc(tmem_holder, 512);  // two accumulator stages, 256 columns apart
    tmem_relinquish();
  }
  if (threadIdx.x >= 64 && threadIdx.x < 64 + kNB) s_bias[threadIdx.x - 64] = p.bias ? p.bias[threadIdx.x - 64] : 0.f;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_holder, 0);
  if (warp == 0) N48_STAMP(1);
  pdl_launch_dependents();

  if (warp == 0) {
    // ===================== TMA producer =====================
    const bool leader = elect_one();
    if (leader) {
      for (int ky = 0; ky < 3; ++ky) {   // one barrier per kernel row: the first MMAs start after a third of the weights
        mbar_expect_tx(&bar_w[ky], kWRow);
        tma_load_2d(smem_w + ky * kWRow, &tmW, &bar_w[ky], 0, ky * 3 * kNB);
      }
    }
    pdl_wait();  // the packed weights are old; the activations come from the previous kernel
    if (warp == 0) N48_STAMP(2);
    int it = 0;
    for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++it) {
      const int slot = it % p.nstage;
      const uint32_t ph = (it / p.nstage) & 1;
      mbar_wait(&bar_empty[slot], ph ^ 1, 1);
      uint8_t* dst = smem_a + slot * p.stage_bytes;
      const int row0 = tile * kNTileOut - 1 - p.P;  // first PTL row kernel row 0 reads
      if (leader) {
        mbar_expect_tx(&bar_full[slot], p.stage_bytes);
        for (int b = 0; b < p.nbox; ++b) tma_load_2d(dst + b * p.box_rows * 128, &tmA, &bar_full[slot], 0, row0 + b * p.box_step);
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    const bool leader = elect_one();
    constexpr uint32_t idesc = make_idesc_bf16(128, 3 * kNB, 0, 0);
    constexpr uint32_t dhi = sdesc_hi_sw128(1024);
    const uint32_t w_lo = sdesc_lo(smem_u32(smem_w), 16);
    const uint32_t a_lo0 = sdesc_lo(smem_u32(smem_a), 16);
    const uint32_t ky_step = uint32_t(p.ky_step16);
    int it = 0;
    for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++it) {
      const int slot = it % p.nstage;
      const uint32_t ph = (it / p.nstage) & 1;
      const int acc = it & 1;
      const uint32_t aph = (it >> 1) & 1;
      long long w0 = 0, w1 = 0;
      if (tl) w0 = clock64();
      mbar_wait(&bar_tempty[acc], aph ^ 1, 3);
      if (tl) w1 = clock64();
      mbar_wait(&bar_full[slot], ph, 4);
      if (tl && lane == 0 && it > 0) { tl[14] += w1 - w0; tl[15] += clock64() - w1; }
      if (it == 0) N48_STAMP(4);
      tc_fence_after();
      const uint32_t a_tile = a_lo0 + uint32_t(slot * p.stage_bytes) / 16;
      const uint32_t d_tmem = tmem_base + uint32_t(acc * 256);
#pragma unroll
      for (int ky = 0; ky < 3; ++ky) {
        if (it == 0) {
          mbar_wait(&bar_w[ky], 0, 2);
          tc_fence_after();
          if (ky == 0) N48_STAMP(3);
        }
        if (leader) {
          const uint32_t a_row = a_tile + uint32_t(ky) * ky_step;
          const uint32_t b_row = w_lo + uint32_t(ky * 3 * kNB * 8);
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            if (ky == 0 && k == 0) umma_bf16_lohi<false>(d_tmem, a_row, dhi, b_row, dhi, idesc);
            else umma_bf16_lohi<true>(d_tmem, a_row + k * 2, dhi, b_row + k * 2, dhi, idesc);
          }
        }
        __syncwarp();
      }
      if (leader) {
        umma_commit(&bar_empty[slot]);  // ring slot free once these MMAs retire
        umma_commit(&bar_tfull[acc]);   // accumulator ready
      }
      __syncwarp();
    }
    N48_STAMP(5);
  } else {
    // ===================== epilogue: 16 columns per tap, planar fp32 output =====================
    const int ew = warp - 2;
    const int grp = ew >> 3;
    const int wq = warp & 3;
    const int RP = p.R * p.P;
    float* xch = reinterpret_cast<float*>(smem + p.off_xch) + grp * 512;
    const int src_up = (lane + 31) & 31, src_dn = (lane + 1) & 31;
    const bool f_relu = bool(p.flags & SRES_EPI_RELU);
    pdl_wait();
    if (((ew >> 2) & 1) == 0) {   // one warp per lane quarter and group; the other eight epilogue warps have nothing to do
      for (int tile = blockIdx.x + grp * gridDim.x, it = grp; tile < p.n_tiles; tile += 2 * gridDim.x, it += 2) {
        const uint32_t aph = (it >> 1) & 1;
        const int tile_base = tile * kNTileOut;
        const int i = wq * 32 + lane;
        const int q = tile_base - 1 + i;
        const bool own = i >= 1 && i <= kNTileOut && q < p.npos;
        const int qc = own ? q : tile_base;
        const int b = qc / RP;
        const int rem = qc - b * RP;
        const int y = rem / p.P;
        const int x = rem - y * p.P;
        const bool live = own && x != p.W && y != p.H;
        mbar_wait(&bar_tfull[grp], aph, 5);
        tc_fence_after();
        uint32_t d0[16], d1[16], d2[16];
        const uint32_t trow = tmem_base + (uint32_t(wq * 32) << 16) + uint32_t(grp * 256);
        tmem_ld16(trow, d0);
        tmem_ld16(trow + 16, d1);
        tmem_ld16(trow + 32, d2);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bar_tempty[grp]);
        float* xs = xch + (it & 2) * 128;   // two slots, alternating per tile of this group
        if (lane == 31) {
          float4* d = reinterpret_cast<float4*>(xs + (0 * 4 + wq) * 16);
#pragma unroll
          for (int j = 0; j < 4; ++j)
            d[j] = make_float4(__uint_as_float(d0[4 * j]), __uint_as_float(d0[4 * j + 1]), __uint_as_float(d0[4 * j + 2]),
                               __uint_as_float(d0[4 * j + 3]));
        }
        if (lane == 0) {
          float4* d = reinterpret_cast<float4*>(xs + (1 * 4 + wq) * 16);
#pragma unroll
          for (int j = 0; j < 4; ++j)
            d[j] = make_float4(__uint_as_float(d2[4 * j]), __uint_as_float(d2[4 * j + 1]), __uint_as_float(d2[4 * j + 2]),
                               __uint_as_float(d2[4 * j + 3]));
        }
        named_bar_sync(1 + grp, 128);
        if (lane == 31 && wq > 0) {
          const float4* s4 = reinterpret_cast<const float4*>(xs + (0 * 4 + wq - 1) * 16);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float4 t = s4[j];
            d0[4 * j] = __float_as_uint(t.x); d0[4 * j + 1] = __float_as_uint(t.y);
            d0[4 * j + 2] = __float_as_uint(t.z); d0[4 * j + 3] = __float_as_uint(t.w);
          }
        }
        if (lane == 0 && wq < 3) {
          const float4* s4 = reinterpret_cast<const float4*>(xs + (1 * 4 + wq + 1) * 16);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float4 t = s4[j];
            d2[4 * j] = __float_as_uint(t.x); d2[4 * j + 1] = __float_as_uint(t.y);
            d2[4 * j + 2] = __float_as_uint(t.z); d2[4 * j + 3] = __float_as_uint(t.w);
          }
        }
        __syncwarp();
        float* dst = p.out_nchw + ((long long)b * p.c_real * p.H + y) * p.W + x;
#pragma unroll
        for (int c = 0; c < 16; ++c) {
          if (c < p.c_real) {   // warp-uniform: only the real output channels are shifted and stored
            const float up = __uint_as_float(__shfl_sync(0xffffffffu, d0[c], src_up));
            const float dn = __uint_as_float(__shfl_sync(0xffffffffu, d2[c], src_dn));
            float v = ((__uint_as_float(d1[c]) + s_bias[c]) + up) + dn;
            if (f_relu) v = fmaxf(v, 0.f);
            if (live) dst[(long long)c * p.H * p.W] = v;   // consecutive lanes = consecutive pixels of a plane
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (tl && threadIdx.x == 0) tl[12] = clock64();
  if (warp == 0) tmem_dealloc(tmem_base, 512);
#undef N48_STAMP
}

// shared-memory plan: weights | ring | exchange | barriers
struct N48Plan {
  int nbox, box_rows, box_step, ky_step16, stage_bytes, nstage;
  int off_xch, off_tail;
  size_t smem;
};
static bool n48_plan(N48Plan* pl, int W) {
  const int smem_max = 232448;  // 227 KB
  const int P = W + 1;
  const int window = 128 + 2 * P;   // union of the three kernel rows' 128-row blocks
  if (window < 3 * 128) {           // one window, split into boxes of <= 256 rows (8-row swizzle atoms)
    pl->nbox = (window + 255) / 256;
    pl->box_rows = ((window + pl->nbox - 1) / pl->nbox + 7) / 8 * 8;
    pl->box_step = pl->box_rows;
    pl->ky_step16 = P * 8;
  } else {                          // wide image: one independent 128-row block per kernel row
    pl->nbox = 3; pl->box_rows = 128; pl->box_step = P; pl->ky_step16 = 128 * 8;
  }
  pl->stage_bytes = pl->nbox * pl->box_rows * 128;
  int ns = (smem_max - 1024 - kNWBytes - 4096 - 1024) / pl->stage_bytes;
  if (ns > kNStages) ns = kNStages;
  if (ns < 2) return false;
  pl->nstage = ns;
  int off = kNWBytes + ns * pl->stage_bytes;
  pl->off_xch = off; off += 4096;
  pl->off_tail = off; off += 1024;
  pl->smem = (size_t)off + 1024;
  return true;
}

// tail convolution 64 -> c_real <= 16 (weights packed with 16 rows per tap), planar fp32 output, any image width
bool conv_n48_available(int H, int W) {
  (void)H;
  N48Plan pl;
  static const int on = [] { const char* e = getenv("SRES_CONV_N48"); return e ? atoi(e) : 1; }();
  return on != 0 && n48_plan(&pl, W);
}

int launch_conv_n48(const sres_conv_args* a, cudaStream_t stream) {
  ConvN48Params p{};
  p.H = a->H; p.W = a->W; p.P = a->W + 1; p.R = a->H + 1;
  const long long npos = (long long)a->B * p.R * p.P;
  if (npos > 0x7fff0000LL) return set_error(SRES_ERR_UNSUPPORTED, "conv: batch too large for 32-bit rows");
  p.npos = (int)npos;
  p.n_tiles = (p.npos + kNTileOut - 1) / kNTileOut;
  p.flags = a->epi_flags; p.bias = a->bias; p.out_nchw = a->out_nchw; p.c_real = a->c_real;
  p.timeline = (long long*)a->debug_timeline;
  N48Plan pl;
  if (!n48_plan(&pl, a->W)) return set_error(SRES_ERR_UNSUPPORTED, "conv: no room for the halo ring");
  p.nstage = pl.nstage; p.stage_bytes = pl.stage_bytes; p.nbox = pl.nbox; p.box_rows = pl.box_rows; p.box_step = pl.box_step;
  p.ky_step16 = pl.ky_step16;
  p.off_xch = pl.off_xch; p.off_tail = pl.off_tail;
  CUtensorMap tmA, tmW;
  int rc = make_tmap_rows64(&tmA, a->in_bf16, (uint64_t)p.npos, pl.box_rows);
  if (rc) return rc;
  rc = make_tmap_rows64(&tmW, a->wpack_bf16, 9 * kNB, 3 * kNB);
  if (rc) return rc;
  const int sms = device_sm_count();
  if (sms <= 0) return set_error(SRES_ERR_NO_DEVICE, "conv: no CUDA device");
  const int grid = persistent_grid(p.n_tiles, sms);
  int dev = 0;
  cudaGetDevice(&dev);
  static thread_local int attr_dev = -1;
  cudaError_t e;
  if (attr_dev != dev) {
    e = cudaFuncSetAttribute(conv3x3_n48_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
    if (e != cudaSuccess) return set_cuda_error(e, "conv: smem attribute");
    attr_dev = dev;
  }
  e = launch_pdl(conv3x3_n48_kernel, dim3(grid), dim3(kNThreads), pl.smem, stream, tmA, tmW, p);
  if (e != cudaSuccess) return set_cuda_error(e, "conv: launch");
  e = cudaGetLastError();
  if (e != cudaSuccess) return set_cuda_error(e, "conv: launch");
  return SRES_OK;
}

}  // namespace sres
