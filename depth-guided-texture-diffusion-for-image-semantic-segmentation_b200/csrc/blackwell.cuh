// sm_100a building blocks written as inline PTX: mbarrier, TMA (cp.async.bulk.tensor),
// tcgen05 (TMEM alloc / mma / commit / ld), UMMA descriptors, tensor-map encoding.
#pragma once
#include <cuda.h>  // CUtensorMap types only; the encoder is fetched through the runtime
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

namespace dgtd {
namespace bw {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ---- mbarrier -------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, 0x989680;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug must surface as a trapped launch, never as a hung GPU.  The bound is WALL time
// (%globaltimer, ns) and generous (20 s): time-slicing, MPS, a debugger or a long preemption stretch a healthy
// wait without advancing the protocol, and must not kill the context.  -DDGTD_NO_MBAR_TRAP removes the trap.
__device__ __forceinline__ unsigned long long global_timer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
#ifdef DGTD_NO_MBAR_TRAP
  while (!mbar_try_wait(bar, parity)) {}
#else
  // the timer is read once per 4096 failed polls (an inner loop without it: written the obvious way, with the read
  // behind `(++spins & 0xfff) == 0`, ptxas speculates the CS2R into every iteration -- 13 instructions per poll, which
  // at 30 M polls per launch of mp_tc_f32_kernel was 40 % of ALL issued instructions, r2 profile)
  const unsigned long long t0 = global_timer_ns();
  for (;;) {
#pragma unroll 1
    for (int i = 0; i < 4096; ++i)
      if (mbar_try_wait(bar, parity)) return;
    if (global_timer_ns() - t0 > 20000000000ULL) {
      printf("dgtd: mbarrier wait timed out after 20 s (block %d thread %d)\n", blockIdx.x, threadIdx.x);
      __trap();
    }
  }
#endif
}

// Wait of a role that has slack: between polls the warp sleeps, so it does not compete for issue slots with the warps
// on the critical path (r2 trace of mp_tc_f32_kernel: with ~12 of 32 warps polling, an instruction of the MMA-issuing
// warp took 10-15 clocks to be selected).
__device__ __forceinline__ void mbar_wait_relaxed(uint64_t* bar, uint32_t parity, unsigned ns) {
  if (mbar_try_wait(bar, parity)) return;
#ifdef DGTD_NO_MBAR_TRAP
  while (!mbar_try_wait(bar, parity)) __nanosleep(ns);
#else
  const unsigned long long t0 = global_timer_ns();
  for (;;) {
#pragma unroll 1
    for (int i = 0; i < 4096; ++i) {
      __nanosleep(ns);
      if (mbar_try_wait(bar, parity)) return;
    }
    if (global_timer_ns() - t0 > 20000000000ULL) {
      printf("dgtd: mbarrier wait timed out after 20 s (block %d thread %d)\n", blockIdx.x, threadIdx.x);
      __trap();
    }
  }
#endif
}

// ---- TMA ------------------------------------------------------------------------------------
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(const CUtensorMap* m, uint64_t* bar, void* dst, int c0,
                                            int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cta.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(const CUtensorMap* m, uint64_t* bar, void* dst, int c0,
                                            int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cta.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1),
      "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_5d(const CUtensorMap* m, uint64_t* bar, void* dst, int c0,
                                            int c1, int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cta.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1),
      "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_5d(const CUtensorMap* m, const void* src, int c0, int c1, int c2, int c3,
                                             int c4) {
  asm volatile("cp.async.bulk.tensor.5d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5, %6}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait_all() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// ---- tcgen05 / TMEM ---------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t cols) {  // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(dst_smem)),
               "r"(cols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t cols) {  // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] . B[smem], bf16 inputs, fp32 accumulate; one thread issues.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                          uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                          uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// mbarrier arrives when all previously issued tcgen05.mma of this thread have completed
// (implies tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   smem_u32(bar))
               : "memory");
}
// 32 lanes x 32 columns of fp32: thread t of the warp gets row (lane base + t), 32 columns.
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]),
        "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]),
        "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]),
        "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- UMMA descriptors -------------------------------------------------------------------------
// K-major operand tile whose rows are `row_bytes` (= swizzle span: 128/64/32 B) long, stored
// densely by TMA with the matching swizzle; 8-row groups are 8*row_bytes apart (SBO).
//   bits [0,14) addr>>4 | [16,30) LBO>>4 (unused for swizzled K-major) | [32,46) SBO>>4 |
//   [46,48) version = 1 (sm_100) | [61,64) layout: 2 = 128B, 4 = 64B, 6 = 32B swizzle
__device__ __forceinline__ uint64_t umma_smem_desc_kmajor(uint32_t smem_addr, uint32_t row_bytes) {
  const uint64_t layout = row_bytes == 128 ? 2ull : row_bytes == 64 ? 4ull : 6ull;
  return (uint64_t)((smem_addr >> 4) & 0x3FFF) | ((uint64_t)((8 * row_bytes) >> 4) << 32) |
         (1ull << 46) | (layout << 61);
}
// MN-major operand, 128-byte swizzle: the tile is stored as K rows of 64 contiguous MN elements
// (128 B, exactly what a {64 MN, k rows} SWIZZLE_128B TMA box writes).  Canonical layout (CUTLASS
// cute/atom/mma_traits_sm100.hpp, "make_umma_desc<Major::MN>", units of 16 B):
//   ((8,n),(8,k)) : ((1,LBO),(8,SBO))   LBO = pitch between 64-element MN blocks,
//                                         SBO = pitch between groups of 8 K rows (1024 B when dense)
__device__ __forceinline__ uint64_t umma_smem_desc_mnmajor_sw128(uint32_t smem_addr, uint32_t lbo_bytes,
                                                                 uint32_t sbo_bytes) {
  return (uint64_t)((smem_addr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | (1ull << 46) | (2ull << 61);
}
// kind::f16 instruction descriptor: fp32 accumulate, bf16 A/B, both K-major, M x N tile
// (bits 15 / 16 set = A / B MN-major).
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// kind::tf32: fp32 accumulator, A / B formats = TF32 (2), K-major both; one instruction covers K = 8 (32 bytes)
__host__ __device__ constexpr uint32_t umma_idesc_tf32(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

}  // namespace bw

// ---- host: tensor-map encoding through the runtime's driver entry point (no -lcuda) ---------
typedef CUresult (*PFN_tmapEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                        const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                        const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                        CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
PFN_tmapEncodeTiled get_tmap_encoder();  // nullptr on failure (error string set)

// rank-`rank` tiled map; dims/box innermost first, strides in bytes for dims 1..rank-1.
int make_tmap(CUtensorMap* out, const void* base, CUtensorMapDataType dt, int rank,
              const uint64_t* dims, const uint64_t* strides_bytes, const uint32_t* box,
              CUtensorMapSwizzle swz);

}  // namespace dgtd
