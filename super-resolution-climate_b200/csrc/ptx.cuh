// Thin inline-PTX wrappers for the sm_100a features the RCAN hot path uses:
// mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld) and
// the UMMA shared-memory + instruction descriptors.  No CUTLASS dependency.
#pragma once
#include <cuda_runtime.h>
#include <cuda.h>
#include <stdint.h>

namespace sres {

// ---------------------------------------------------------------------------
// misc
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}\n"
      : "=r"(pred));
  return pred != 0;
}

// Device-side error word (set before a trap so the host can tell a pipeline
// time-out from other faults).
__device__ unsigned int g_sres_dev_error = 0;

// ---------------------------------------------------------------------------
// programmatic dependent launch: the next kernel of the stream may start its prologue (barrier init,
// TMEM allocation, weight loads) while this one drains; it must pdl_wait() before touching anything a
// predecessor wrote.  Every kernel launched with the attribute calls pdl_wait() on every exit path.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ---------------------------------------------------------------------------
// mbarrier
// ---------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P1;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P1;\n\t}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a broken pipeline traps (launch failure) instead of hanging
// the GPU.  ~4 s at 2 GHz.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, int who = 0) {
  if (mbar_try_wait(bar, parity)) return;
  long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 8000000000LL) {
      atomicExch(&g_sres_dev_error, 0xDEAD0000u | (unsigned)who);
      __threadfence_system();
      __trap();
    }
  }
}

// ---------------------------------------------------------------------------
// TMA
// ---------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar,
                                            int32_t c0, int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0),
        "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* m, uint64_t* bar,
                                            int32_t c0, int32_t c1, int32_t c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5}], [%2];"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0),
        "r"(c1), "r"(c2)
      : "memory");
}
// shared -> global tile store (bulk async group completion)
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* smem_src, int32_t c0, int32_t c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               :
               : "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// wait until at most N of this thread's bulk groups still READ their shared-memory source
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void bulk_wait_all() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}
// generic-proxy writes -> visible to the async proxy (UMMA / TMA store)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ---------------------------------------------------------------------------
// tcgen05: TMEM allocation
// ---------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_holder, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_holder)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// ---------------------------------------------------------------------------
// tcgen05: MMA (kind::f16, bf16 x bf16 -> fp32), one CTA
// ---------------------------------------------------------------------------
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                          uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
      :
      : "r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Same, with the two 64-bit shared-memory descriptors passed as (lo, hi) halves so the issuing thread only
// does one 32-bit add per operand per MMA (the hi halves are loop constants).  The single MMA-issuing
// thread must sustain one instruction per ~32 tensor-pipe cycles; descriptor arithmetic is its bottleneck.
template <bool kAccumulate>
__device__ __forceinline__ void umma_bf16_lohi(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo,
                                               uint32_t b_hi, uint32_t idesc) {
  if constexpr (kAccumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
        "mov.b64 da, {%1, %2};\n\tmov.b64 db, {%3, %4};\n\t"
        "setp.eq.b32 p, 0, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}\n"
        :
        : "r"(tmem_d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc)
        : "memory");
  } else {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
        "mov.b64 da, {%1, %2};\n\tmov.b64 db, {%3, %4};\n\t"
        "setp.ne.b32 p, 0, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}\n"
        :
        : "r"(tmem_d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc)
        : "memory");
  }
}
__device__ __forceinline__ void umma_bf16_lohi_p(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo,
                                                 uint32_t b_hi, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %2};\n\tmov.b64 db, {%3, %4};\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}\n"
      :
      : "r"(tmem_d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
// hi / lo halves of a SWIZZLE_128B descriptor (see make_sdesc_sw128)
__device__ __forceinline__ constexpr uint32_t sdesc_hi_sw128(uint32_t sbo_bytes) {
  return ((sbo_bytes >> 4) & 0x3FFF) | (1u << 14) | (2u << 29);
}
__device__ __forceinline__ uint32_t sdesc_lo(uint32_t saddr, uint32_t lbo_bytes) {
  return ((saddr >> 4) & 0x3FFF) | (((lbo_bytes >> 4) & 0x3FFF) << 16);
}
// Ampere-style asynchronous 4-byte copy global -> shared; src_bytes == 0 writes zeros without touching global memory.
__device__ __forceinline__ void cp_async4_zfill(void* smem_dst, const void* gsrc, int src_bytes) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// Packed fp32 FMA (sm_100: FFMA2): acc.{x,y} = fma(a.{x,y}, s, acc.{x,y}), each half rounded like fmaf.  ptxas folds the
// duplicated scalar into the instruction's broadcast operand form (FFMA2 Rd, Ra.F32x2, Rs.F32, Rd.F32x2), so one issue slot
// does two FMAs -- the CUDA-core convolutions at the network's two ends are issue-bound, not HBM-bound.
__device__ __forceinline__ void ffma2_bcast(float2& acc, const float2& a, float s) {
  const float2 ss = make_float2(s, s);
  asm("fma.rn.f32x2 %0, %1, %2, %0;"
      : "+l"(reinterpret_cast<uint64_t&>(acc))
      : "l"(reinterpret_cast<const uint64_t&>(a)), "l"(reinterpret_cast<const uint64_t&>(ss)));
}

// Arrive on an mbarrier once all previously issued MMAs of this thread retire.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   smem_u32(bar))
               : "memory");
}

// Instruction descriptor for kind::f16: bf16 A/B, fp32 D.
//   bits [4,6) c_format (1 = F32); [7,10) a_format (1 = BF16); [10,13) b_format;
//   bit 15 a_major (0 = K, 1 = MN); bit 16 b_major; [17,23) N>>3; [24,29) M>>4.
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N, int a_mn_major,
                                                       int b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (uint32_t(a_mn_major) << 15) |
         (uint32_t(b_mn_major) << 16) | (uint32_t(N >> 3) << 17) | (uint32_t(M >> 4) << 24);
}

// Shared-memory matrix descriptor, SWIZZLE_128B.
//   [0,14) start>>4; [16,30) LBO>>4; [32,46) SBO>>4; [46,48) version = 1;
//   [49,52) base_offset; [61,64) layout type (2 = SWIZZLE_128B).
// Every operand tile in this project is stored as rows of 128 B (64 bf16), row r at
// base + 128*r, 16-byte chunks XOR-swizzled by (r & 7) -- exactly what a TMA load with
// CU_TENSOR_MAP_SWIZZLE_128B produces for a 1024-B-aligned destination.
//   K-major use  (row = M/N index, 64 K elements per row): SBO = 1024 (8 rows), LBO unused.
//   MN-major use (row = K index, 64 M/N elements per row): SBO = 1024 (8 k-rows),
//                LBO = byte distance to the next group of 64 M/N elements.
__device__ __forceinline__ uint64_t make_sdesc_sw128(uint32_t saddr, uint32_t lbo_bytes,
                                                     uint32_t sbo_bytes, uint32_t base_offset) {
  uint64_t d = 0;
  d |= uint64_t((saddr >> 4) & 0x3FFF);
  d |= uint64_t((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= uint64_t((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= uint64_t(1) << 46;
  d |= uint64_t(base_offset & 7) << 49;
  d |= uint64_t(2) << 61;
  return d;
}

// ---------------------------------------------------------------------------
// tcgen05: TMEM -> registers.  32 lanes x 32 bit x 16 columns per warp.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
        "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
        "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
// 16 lanes x 256 bit, repeated 4x along the columns (32 columns): the accumulator-fragment layout -- thread t
// gets rows t/4 and t/4+8 of the 16-lane group, columns 8k + 2(t%4) + {0,1}: v[4k + 2h + e] = D[t/4 + 8h][8k + 2(t%4) + e].
// Column reductions over the rows then need 3 shuffle stages on 8 values instead of 5 stages on 32.
__device__ __forceinline__ void tmem_ld_frag16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.16x256b.x4.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
        "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
        "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// ---------------------------------------------------------------------------
// small helpers
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ float bf16_lo(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t v) { return __uint_as_float(v & 0xFFFF0000u); }

}  // namespace sres
