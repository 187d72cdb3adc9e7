// Weight gradient of the 3x3 / 64-feature convolution as a split-K tcgen05 GEMM (sm_100a).
//
//   dW[tap][ci][co] = sum_q  X[q + off(tap)][ci] * dY[q][co]          q = PTL row (the K dimension)
//
// Both operands are "MN-major": a shared-memory row is one K index (position) holding 64 contiguous
// channels -- exactly the PTL row the TMA loads.  Two taps are stacked on the UMMA M dimension
// (M = 128 = 2 x 64 ci): the second group of 64 rows is the SAME halo window shifted by
// (off_b - off_a) rows, expressed through the descriptor's leading-dimension byte offset.  9 taps
// -> 5 accumulators of 128 x 64 fp32 in TMEM (the last one carries one junk half).
//
// N128 variant (opt-in, see wgrad_n128_enabled): the SAME stacking trick on the N side.  The MMA's K index k pairs X[k + alpha] with
// dY[k + beta], which is the tap of offset alpha - beta; two dY windows (beta = -P and 0, second 64-column group
// reached through the B descriptor's leading-dimension offset) times two X windows give FOUR taps per
// M128 x N128 MMA:  {-P-1,-P} x {-P,0} -> taps (1,0)(1,1)(0,0)(0,1);  {-P+1,+1} x {-P,0} -> (1,2)(2,2)(0,2)(dup);
// {P-1,P} x {0} -> (2,0)(2,1) (N = 64).  3 MMA groups instead of 5 per K step, 22 KB instead of 30 KB of operand
// reads from shared memory -- the resource that bounds this kernel.  (dY's padding rows are zero, so the rows the
// shifted window drops at the very end of the buffer contribute nothing.)
//
// Up to SRES_WGRAD_MAX_JOBS (8) independent weight gradients ("jobs": different layers of the backward pass) share one
// launch: CTA c works on job c % njobs and reduces every nsplit-th 128-position chunk of it.  Fewer
// split-K partials per job means less partial traffic and the per-launch cost (prologue, accumulator
// drain) is paid once per batch.  Each CTA TMA-stores its fp32 partial [5][128][64] (+ the bias-gradient
// partial, column sums of dY); a second kernel sums the partials in a fixed order (deterministic) and
// scatters them into the OIHW fp32 gradient.
//
// Replaces the weight/bias part of aten::convolution_backward for the reference's nn.Conv2d
// (sres/model/common/cnn.py:8-9), reached from mloss.backward() (dual_trainer.py:322).
#include "ptx.cuh"
#include "internal.h"

namespace sres {

constexpr int kWgMaxStages = 4;
constexpr int kWgAcc = 5;
constexpr int kWgMaxJobs = SRES_WGRAD_MAX_JOBS;
constexpr int kWgPartFloats = kWgAcc * 128 * 64;  // one partial: [5][128][64]

struct WgMaps {
  CUtensorMap x[kWgMaxJobs];
  CUtensorMap dy[kWgMaxJobs];
};

struct WgradKParams {
  int P, npos, n_chunks, nstage, xrows, dyrows, njobs, max_split;
  int xbox, dybox;     // rows per TMA box of the X window / the dY tile (the tensor maps are encoded with these)
  int off_a[kWgAcc];   // row offset (ky*P+kx) of the first tap of each accumulator
  int lbo[kWgAcc];     // byte distance to the second tap's window
  float* part_bias;    // [njobs][max_split][64]
};

template <bool N128>
__global__ void __launch_bounds__(256, 1)
conv3x3_wgrad_kernel(const __grid_constant__ WgMaps maps, const __grid_constant__ CUtensorMap tmPart, const WgradKParams p) {
  extern __shared__ uint8_t smem_raw[];
  // offset arithmetic (not an integer round trip) keeps the pointer in the shared address space: LDS/STS, not generic LD/ST
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int stage_bytes = (p.dyrows + p.xrows) * 128;
  const int dy_row0 = N128 ? p.P : 0;   // window row of PTL row q0 (the window starts P rows earlier for the beta = -P group)
  uint8_t* tail = smem + p.nstage * stage_bytes;
  uint64_t* bar_full = reinterpret_cast<uint64_t*>(tail);
  uint64_t* bar_empty = bar_full + kWgMaxStages;
  uint64_t* bar_done = bar_empty + kWgMaxStages;
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(bar_done + 1);
  float* s_db = reinterpret_cast<float*>(tmem_holder + 2);  // [4][64]

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);  // warp-uniform by construction
  const int lane = threadIdx.x & 31;
  // this CTA's job and its position among the CTAs of that job
  const int job = blockIdx.x % p.njobs;
  const int split = blockIdx.x / p.njobs;
  const int nsplit = (int(gridDim.x) - job + p.njobs - 1) / p.njobs;
  const CUtensorMap* tmX = &maps.x[job];
  const CUtensorMap* tmDY = &maps.dy[job];

  if (threadIdx.x == 0) {
    tma_prefetch_desc(tmX);
    tma_prefetch_desc(tmDY);
    for (int i = 0; i < kWgMaxStages; ++i) {
      mbar_init(&bar_full[i], 1);
      mbar_init(&bar_empty[i], 1 + 4);  // MMA commit + 4 bias-gradient warps
    }
    mbar_init(bar_done, 1);
    mbar_fence_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_holder, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_holder, 0);
  pdl_launch_dependents();

  if (warp == 0) {
    const bool leader = elect_one();
    pdl_wait();
    int it = 0;
    for (int c = split; c < p.n_chunks; c += nsplit, ++it) {
      const int slot = it % p.nstage;
      const uint32_t ph = (it / p.nstage) & 1;
      mbar_wait(&bar_empty[slot], ph ^ 1, 11);
      uint8_t* dst = smem + slot * stage_bytes;
      const int q0 = c * 128;
      if (leader) {
        mbar_expect_tx(&bar_full[slot], stage_bytes);
        for (int r = 0; r < p.dyrows; r += p.dybox) tma_load_2d(dst + r * 128, tmDY, &bar_full[slot], 0, q0 - dy_row0 + r);
        uint8_t* xdst = dst + p.dyrows * 128;
        const int x0 = q0 - (p.P + 1);
        for (int r = 0; r < p.xrows; r += p.xbox) tma_load_2d(xdst + r * 128, tmX, &bar_full[slot], 0, x0 + r);
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    const bool leader = elect_one();
    constexpr uint32_t idesc = make_idesc_bf16(128, 64, 1, 1);
    constexpr uint32_t idesc128 = make_idesc_bf16(128, 128, 1, 1);
    constexpr uint32_t dhi = sdesc_hi_sw128(1024);
    const uint32_t s_addr = smem_u32(smem);
    uint32_t xoff[kWgAcc];
#pragma unroll
    for (int a = 0; a < kWgAcc; ++a) xoff[a] = uint32_t(p.off_a[a]) * 8 + ((uint32_t(p.lbo[a]) >> 4) << 16);
    int it = 0;
    for (int c = split; c < p.n_chunks; c += nsplit, ++it) {
      const int slot = it % p.nstage;
      const uint32_t ph = (it / p.nstage) & 1;
      mbar_wait(&bar_full[slot], ph, 12);
      tc_fence_after();
      const uint32_t x_lo = sdesc_lo(s_addr + slot * stage_bytes + p.dyrows * 128, 0);
      if (leader) {
        if constexpr (N128) {
          // B: dY window rows [q0 - P, ...): column group 0 = beta -P (window row k), group 1 = beta 0 (row k + P)
          const uint32_t dy2_lo = sdesc_lo(s_addr + slot * stage_bytes, uint32_t(p.P) * 128);
          const uint32_t dy1_lo = sdesc_lo(s_addr + slot * stage_bytes + p.P * 128, 1024);
#pragma unroll
          for (int g = 0; g < 3; ++g) {
            const uint32_t xa = x_lo + xoff[g];
            const uint32_t dcol = tmem_base + g * 128;
#pragma unroll
            for (int kk = 0; kk < 8; ++kk) {
              if (g < 2) {
                if (kk == 0) umma_bf16_lohi_p(dcol, xa, dhi, dy2_lo, dhi, idesc128, it ? 1u : 0u);
                else umma_bf16_lohi<true>(dcol, xa + kk * 128, dhi, dy2_lo + kk * 128, dhi, idesc128);
              } else {
                if (kk == 0) umma_bf16_lohi_p(dcol, xa, dhi, dy1_lo, dhi, idesc, it ? 1u : 0u);
                else umma_bf16_lohi<true>(dcol, xa + kk * 128, dhi, dy1_lo + kk * 128, dhi, idesc);
              }
            }
          }
        } else {
          const uint32_t dy_lo = sdesc_lo(s_addr + slot * stage_bytes, 1024);
#pragma unroll
          for (int a = 0; a < kWgAcc; ++a) {
            const uint32_t xa = x_lo + xoff[a];
#pragma unroll
            for (int kk = 0; kk < 8; ++kk) {
              if (kk == 0) umma_bf16_lohi_p(tmem_base + a * 64, xa, dhi, dy_lo, dhi, idesc, it ? 1u : 0u);
              else umma_bf16_lohi<true>(tmem_base + a * 64, xa + kk * 128, dhi, dy_lo + kk * 128, dhi, idesc);
            }
          }
        }
        umma_commit(&bar_empty[slot]);
      }
      __syncwarp();
    }
    if (leader) umma_commit(bar_done);
  } else if (warp >= 4) {
    // bias gradient: column sums of the dY tile, read straight from the swizzled smem rows.
    // 128-bit loads: lane = (row group rg = lane / 8, 16-byte chunk ck = lane % 8) -> 4 rows per instruction,
    // 8 instructions per 32-row slice; the 4 row groups are folded once at the end.
    const int wq = warp & 3;
    const int rg = lane >> 3, ck = lane & 7;
    float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};  // channels 8*ck .. 8*ck+7
    pdl_wait();  // the partial buffers this CTA overwrites may still be read by the previous batch's reduce
    int it = 0;
    for (int c = split; c < p.n_chunks; c += nsplit, ++it) {
      const int slot = it % p.nstage;
      const uint32_t ph = (it / p.nstage) & 1;
      mbar_wait(&bar_full[slot], ph, 13);
      const uint8_t* dy = smem + slot * stage_bytes;
#pragma unroll
      for (int r = 0; r < 32; r += 4) {
        const int row = dy_row0 + wq * 32 + r + rg;
        const uint4 v = *reinterpret_cast<const uint4*>(dy + row * 128 + ((ck ^ (row & 7)) << 4));
        acc[0] += bf16_lo(v.x); acc[1] += bf16_hi(v.x); acc[2] += bf16_lo(v.y); acc[3] += bf16_hi(v.y);
        acc[4] += bf16_lo(v.z); acc[5] += bf16_hi(v.z); acc[6] += bf16_lo(v.w); acc[7] += bf16_hi(v.w);
      }
      // The arrive hands the slot back to the TMA producer (async proxy).  These generic-proxy loads must be ordered
      // before it by a PROXY fence: without it ptxas schedules the arrive ahead of the last loads' consumers, and under
      // load-store pressure from co-resident kernels the refill overtook a load (one conv-bias gradient off by ~0.5 % in
      // a fraction of the backward passes; tests/test_gpu_model.py::test_full_size_properties).
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_empty[slot]);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], 8);
      acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], 16);
    }
    if (rg == 0) {
#pragma unroll
      for (int j = 0; j < 8; ++j) s_db[wq * 64 + 8 * ck + j] = acc[j];
    }
    asm volatile("bar.sync 1, 128;" ::: "memory");  // all four warps are done reading the operand ring
    // drain the accumulators: TMEM -> swizzled smem slab (the operand ring is idle now) -> TMA store
    mbar_wait(bar_done, 0, 14);
    tc_fence_after();
    uint8_t* slab = smem + wq * 8192;  // [2 halves][32 rows x 128 B]
    const int sw7 = lane & 7;
    const int prow0 = ((job * p.max_split + split) * kWgAcc) * 128 + wq * 32;  // row of the partial matrix
    for (int a = 0; a < kWgAcc; ++a) {
      if (lane == 0) bulk_wait_read<0>();
      __syncwarp();
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        uint32_t raw[32];
        tmem_ld32(tmem_base + (uint32_t(wq * 32) << 16) + a * 64 + h * 32, raw);
        tmem_ld_wait();
        uint8_t* row = slab + h * 4096 + lane * 128;
#pragma unroll
        for (int j = 0; j < 8; ++j)
          *reinterpret_cast<float4*>(row + ((j ^ sw7) << 4)) =
              make_float4(__uint_as_float(raw[4 * j]), __uint_as_float(raw[4 * j + 1]), __uint_as_float(raw[4 * j + 2]),
                          __uint_as_float(raw[4 * j + 3]));
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        tma_store_2d(&tmPart, slab, 0, prow0 + a * 128);
        tma_store_2d(&tmPart, slab + 4096, 32, prow0 + a * 128);
        bulk_commit();
      }
    }
    if (lane == 0) bulk_wait_all<0>();
  }
  tc_fence_before();
  __syncthreads();
  if (threadIdx.x < 64) {
    float* out = p.part_bias + ((size_t)job * p.max_split + split) * 64;
    out[threadIdx.x] = s_db[threadIdx.x] + s_db[64 + threadIdx.x] + s_db[128 + threadIdx.x] + s_db[192 + threadIdx.x];
  }
  if (warp == 2) tmem_dealloc(tmem_base, 512);
}

// Sum the per-CTA partials in split order and scatter into the OIHW gradient.
//   accumulator a, row m = half*64 + ci, column n = co   ->  tap = 2a + half (a < 4), tap 8 for a == 4 half 0
struct WgReduceJob {
  float* dw;
  float* db;
  int cout_total, oc_stride, oc_offset, accumulate, nsplit;
  float scale;
};
struct WgReduceJobs {
  WgReduceJob j[kWgMaxJobs];
  signed char tap[2 * kWgAcc];  // tap held by (64-column block a, row half h) of the partial, -1 = junk / duplicate
};

// Every thread sums FOUR consecutive output features of one (accumulator block, row) over the split-K partials with 16-byte
// loads, eight partials in flight at a time (the first version: one float per thread, one load in flight: 8.9 us per batch of
// four jobs = 2.7 TB/s on data that mostly still sits in L2).  The summation order is fixed -- partials 0, 1, 2, ... into one
// accumulator per feature -- so the result is bit-identical to the scalar version and reproducible run to run.
__global__ void __launch_bounds__(256)
wgrad_reduce_kernel(const float* __restrict__ part, const float* __restrict__ part_bias, int max_split,
                    const __grid_constant__ WgReduceJobs jobs) {
  pdl_wait();
  pdl_launch_dependents();
  const int job = blockIdx.y;
  const WgReduceJob& J = jobs.j[job];
  const int idx4 = blockIdx.x * blockDim.x + threadIdx.x;   // group of four floats
  constexpr int kGroups = kWgPartFloats / 4;
  if (idx4 >= kGroups + 16) return;
  if (idx4 >= kGroups) {   // bias: 16 threads x 4 features
    const int co0 = (idx4 - kGroups) * 4;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int i = 0; i < J.nsplit; ++i) {
      const float4 v = *reinterpret_cast<const float4*>(part_bias + ((size_t)job * max_split + i) * 64 + co0);
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
    const float r[4] = {s.x * J.scale, s.y * J.scale, s.z * J.scale, s.w * J.scale};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int oc = (co0 + e) * J.oc_stride + J.oc_offset;
      if (J.db && oc < J.cout_total) J.db[oc] = J.accumulate ? J.db[oc] + r[e] : r[e];
    }
    return;
  }
  const int idx = idx4 * 4;
  const float4* pp = reinterpret_cast<const float4*>(part + (size_t)job * max_split * kWgPartFloats + idx);
  constexpr size_t kStride4 = kWgPartFloats / 4;
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  int i = 0;
  for (; i + 8 <= J.nsplit; i += 8) {
    float4 v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) v[u] = pp[(size_t)(i + u) * kStride4];
#pragma unroll
    for (int u = 0; u < 8; ++u) { s.x += v[u].x; s.y += v[u].y; s.z += v[u].z; s.w += v[u].w; }
  }
  for (; i < J.nsplit; ++i) {
    const float4 v = pp[(size_t)i * kStride4];
    s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
  }
  const int n0 = idx & 63;
  const int m = (idx >> 6) & 127;
  const int a = idx >> 13;
  const int half = m >> 6, ci = m & 63;
  const int tap = jobs.tap[2 * a + half];
  if (tap < 0) return;
  const float r[4] = {s.x * J.scale, s.y * J.scale, s.z * J.scale, s.w * J.scale};
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const int oc = (n0 + e) * J.oc_stride + J.oc_offset;
    if (oc >= J.cout_total) continue;
    float* o = J.dw + ((size_t)oc * 64 + ci) * 9 + tap;
    *o = J.accumulate ? *o + r[e] : r[e];
  }
}

// Opt-in (SRES_WGRAD_N128=1, read per call so tests can flip it): measured on B200 the four-taps-per-MMA scheme is
// NOT faster than the plain one (33.6 vs 31.1 us per job alone, 29.1 vs 29.0 ms per step) although it reads 27 % fewer
// operand bytes -- the N = 128 MN-major B operand does not stream out of shared memory as well as two N = 64 ones.
static bool wgrad_n128_enabled() {
  const char* e = getenv("SRES_WGRAD_N128");
  return e && atoi(e) != 0;
}

static int wg_grid() {
  int sms = device_sm_count();
  return sms > 0 ? sms : 148;
}

}  // namespace sres

using namespace sres;

extern "C" size_t sres_conv_wgrad_workspace_bytes(void) {
  // partial matrix for a full grid of CTAs (+ one spare per job for rounding) and the bias partials
  const size_t slots = (size_t)wg_grid() + kWgMaxJobs;
  return slots * kWgPartFloats * sizeof(float) + slots * 64 * sizeof(float) + 1024;
}

extern "C" int sres_conv3x3_wgrad_batch(const sres_wgrad_job* jobs, int njobs, int B, int H, int W, void* workspace,
                                        size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (!jobs || njobs < 1 || njobs > kWgMaxJobs) return set_error(SRES_ERR_INVALID_ARG, "wgrad: 1..8 jobs per batch");
  if (!workspace) return set_error(SRES_ERR_INVALID_ARG, "wgrad: null workspace");
  if (B <= 0 || H <= 0 || W <= 0) return set_error(SRES_ERR_INVALID_ARG, "wgrad: bad geometry");
  // Checked before anything touches the device: with oc_stride 0 the reduce's 64 threads of a row would race on one
  // element, and an offset outside [0, oc_stride) would write into another sub-convolution's rows.
  for (int j = 0; j < njobs; ++j) {
    const sres_wgrad_job& J = jobs[j];
    if (!J.x_bf16 || !J.dy_bf16 || !J.dw_oihw) return set_error(SRES_ERR_INVALID_ARG, "wgrad: null pointer in job");
    if (J.cout_total < 1 || J.oc_stride < 1 || J.oc_offset < 0 || J.oc_offset >= J.oc_stride)
      return set_error(SRES_ERR_INVALID_ARG, "wgrad: need cout_total >= 1, oc_stride >= 1 and 0 <= oc_offset < oc_stride");
  }
  WgradKParams p{};
  p.P = W + 1;
  const long long npos = (long long)B * (H + 1) * (W + 1);
  if (npos > 0x7fffff00LL) return set_error(SRES_ERR_UNSUPPORTED, "wgrad: batch too large");
  p.npos = (int)npos;
  p.n_chunks = (p.npos + 127) / 128;
  // X window: 128 positions + the halo of 2(P+1)+1 rows.  When it fits one TMA box (<= 256 rows) it is loaded exactly
  // (rounded to the 8-row swizzle period) in ONE copy; wider windows go in 64-row boxes.  The kernel's slope per job is set
  // by this feed, not by its MMAs (see wgrad_n128_enabled), so the 24 rows the 64-row rounding added at 48 x 48 were 6 % of it.
  const int xneed = 128 + 2 * (p.P + 1) + 1;
  bool n128 = wgrad_n128_enabled();
  const bool exact = !n128 && (xneed + 7) / 8 * 8 <= 256 && !getenv("SRES_WGRAD_BOX64");
  p.xrows = exact ? (xneed + 7) / 8 * 8 : (xneed + 63) / 64 * 64;
  p.xbox = exact ? p.xrows : 64;
  p.dybox = exact ? 128 : 64;
  p.dyrows = n128 ? (128 + p.P + 63) / 64 * 64 : 128;
  if (n128 && ((232448 - 1024 - 2048) / ((p.dyrows + p.xrows) * 128) < 1 || p.P * 128 >= (1 << 18))) {
    n128 = false;  // very wide images: the plain scheme needs less shared memory
    p.dyrows = 128;
  }
  const int stage_bytes = (p.dyrows + p.xrows) * 128;
  int nstage = (232448 - 1024 - 2048) / stage_bytes;
  if (nstage > kWgMaxStages) nstage = kWgMaxStages;
  if (nstage < 1) return set_error(SRES_ERR_UNSUPPORTED, "wgrad: image too wide for the flat halo window");
  if (nstage * stage_bytes < 32768) return set_error(SRES_ERR_UNSUPPORTED, "wgrad: operand ring smaller than the drain slabs");
  p.nstage = nstage;
  WgReduceJobs rj;
  if (n128) {
    // X-window row offsets (window starts at q0 - P - 1) and second-half distances of the three MMA groups
    const int offs[3] = {0, 2, 2 * p.P}, lbos[3] = {128, p.P * 128, 128};
    for (int g = 0; g < kWgAcc; ++g) { p.off_a[g] = g < 3 ? offs[g] : 0; p.lbo[g] = g < 3 ? lbos[g] : 128; }
    // partial column block a = (group, dY shift): tap offset = alpha - beta (see the header comment)
    const signed char taps[2 * kWgAcc] = {3, 4, 0, 1, 5, 8, 2, -1, 6, 7};
    for (int i = 0; i < 2 * kWgAcc; ++i) rj.tap[i] = taps[i];
  } else {
    for (int a = 0; a < kWgAcc; ++a) {
      const int ta = 2 * a, tb = (2 * a + 1 <= 8) ? 2 * a + 1 : -1;
      const int offa = (ta / 3) * p.P + (ta % 3);
      p.off_a[a] = offa;
      p.lbo[a] = tb >= 0 ? (((tb / 3) * p.P + (tb % 3)) - offa) * 128 : 128;
      if (p.lbo[a] >= (1 << 18)) return set_error(SRES_ERR_UNSUPPORTED, "wgrad: tap distance exceeds descriptor range");
      rj.tap[2 * a] = (signed char)ta;
      rj.tap[2 * a + 1] = (signed char)tb;
    }
  }
  const int sms = device_sm_count();
  if (sms <= 0) return set_error(SRES_ERR_NO_DEVICE, "wgrad: no CUDA device");
  int grid = sms;
  if (grid > p.n_chunks * njobs) grid = p.n_chunks * njobs;
  if (grid < njobs) grid = njobs;
  p.njobs = njobs;
  p.max_split = (grid + njobs - 1) / njobs;
  const size_t part_bytes = (size_t)njobs * p.max_split * kWgPartFloats * sizeof(float);
  const size_t bias_bytes = (size_t)njobs * p.max_split * 64 * sizeof(float);
  if (workspace_bytes < part_bytes + bias_bytes) return set_error(SRES_ERR_INVALID_ARG, "wgrad: workspace too small");
  float* part = (float*)workspace;
  p.part_bias = (float*)((uint8_t*)workspace + part_bytes);

  WgMaps maps;
  for (int j = 0; j < kWgMaxJobs; ++j) {
    const sres_wgrad_job& J = jobs[j < njobs ? j : 0];
    int rc = make_tmap_rows64(&maps.x[j], J.x_bf16, (uint64_t)p.npos, (uint32_t)p.xbox);
    if (rc) return rc;
    rc = make_tmap_rows64(&maps.dy[j], J.dy_bf16, (uint64_t)p.npos, (uint32_t)p.dybox);
    if (rc) return rc;
    rj.j[j].dw = J.dw_oihw; rj.j[j].db = J.dbias; rj.j[j].cout_total = J.cout_total; rj.j[j].oc_stride = J.oc_stride;
    rj.j[j].oc_offset = J.oc_offset; rj.j[j].accumulate = J.accumulate;
    rj.j[j].scale = J.scale;
    rj.j[j].nsplit = j < njobs ? (grid - j + njobs - 1) / njobs : 0;
  }
  CUtensorMap tmPart;
  int rc = make_tmap_rows64_f32(&tmPart, part, (uint64_t)njobs * p.max_split * kWgAcc * 128, 32);
  if (rc) return rc;
  const size_t smem = (size_t)nstage * stage_bytes + 1024 + 2048;
  cudaError_t e = cudaFuncSetAttribute(n128 ? conv3x3_wgrad_kernel<true> : conv3x3_wgrad_kernel<false>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return set_cuda_error(e, "wgrad: smem attribute");
  e = n128 ? launch_pdl(conv3x3_wgrad_kernel<true>, dim3(grid), dim3(256), smem, stream, maps, tmPart, p)
           : launch_pdl(conv3x3_wgrad_kernel<false>, dim3(grid), dim3(256), smem, stream, maps, tmPart, p);
  if (e != cudaSuccess) return set_cuda_error(e, "wgrad: launch");
  const int total = kWgPartFloats / 4 + 16;   // groups of four floats + 16 bias groups
  e = launch_pdl(wgrad_reduce_kernel, dim3((total + 255) / 256, njobs), dim3(256), 0, stream, (const float*)part,
                 (const float*)p.part_bias, p.max_split, rj);
  if (e != cudaSuccess) return set_cuda_error(e, "wgrad: reduce launch");
  return SRES_OK;
}

extern "C" int sres_conv3x3_wgrad(const void* x_bf16, const void* dy_bf16, int B, int H, int W, float* dw_oihw,
                                  float* dbias, int cout_total, int oc_stride, int oc_offset, int accumulate,
                                  void* workspace, size_t workspace_bytes, void* stream) {
  sres_wgrad_job j;
  j.x_bf16 = x_bf16; j.dy_bf16 = dy_bf16; j.dw_oihw = dw_oihw; j.dbias = dbias;
  j.cout_total = cout_total; j.oc_stride = oc_stride; j.oc_offset = oc_offset; j.accumulate = accumulate;
  j.scale = 1.f;
  return sres_conv3x3_wgrad_batch(&j, 1, B, H, W, workspace, workspace_bytes, stream);
}
