// Thin inline-PTX wrappers for the sm_100a features the attention kernels use: mbarrier, TMA
// (cp.async.bulk.tensor), tcgen05 (MMA / TMEM alloc / ld / st / commit / fences) and descriptor builders.
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace svae {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(pred));
  return pred != 0;
}

// ---- mbarrier ------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P;\n\tmbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\tselp.u32 %0, 1, 0, P;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug traps (-> CUDA error on the host) instead of hanging the GPU.  Kept inline and
// minimal (no printf): an out-of-line slow path makes ptxas ignore setmaxnreg and spill the softmax registers.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  // try_wait suspends the thread for a hardware-defined interval by itself; the clock (expensive to read, and a
  // serialising instruction) is only consulted once a wait has lasted far longer than any legitimate one
#pragma unroll 1
  for (int i = 0; i < 4096; ++i)
    if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) __trap();     // ~2 s at 2 GHz
  }
}

// One arrival per warp (called by all 32 lanes, warp-uniform argument): __syncwarp() extends the release of the
// arriving lane to the other lanes' earlier writes.  (Measured the other way round for WAITS: one polling lane per
// warp followed by __syncwarp() is 3.5x SLOWER than all 32 lanes executing try_wait convergently -- the hardware
// suspends a convergent warp, a single-lane loop spins through divergence barriers.)
__device__ __forceinline__ void mbar_arrive_warp(uint64_t* bar) {
  __syncwarp();
  if ((threadIdx.x & 31) == 0) mbar_arrive(bar);
}

// ---- TMA -----------------------------------------------------------------------------------------
__device__ __forceinline__ void prefetch_tensormap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, const void* smem_src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.tile.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(map)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// ---- tcgen05: TMEM management ----------------------------------------------------------------------
template <int COLS>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)), "n"(COLS)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(COLS) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// all previously issued tcgen05.mma of this thread arrive on `bar` when complete
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// D[tmem] (+)= A[smem] * B[smem]
__device__ __forceinline__ void mma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]
__device__ __forceinline__ void mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// ---- tcgen05.ld / st, shape 32x32b: thread i of the warp <-> TMEM lane (base + i), N consecutive 32-bit columns
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}

#define SVAE_DEP8(r, o) "+r"(r[o]), "+r"(r[o + 1]), "+r"(r[o + 2]), "+r"(r[o + 3]), "+r"(r[o + 4]), "+r"(r[o + 5]), "+r"(r[o + 6]), "+r"(r[o + 7])
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
      : "memory");
}
// Ties two 16-register tcgen05.ld results to the wait.
__device__ __forceinline__ void tmem_wait_ld16(uint32_t (&a)[16], uint32_t (&b)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;" : SVAE_DEP8(a, 0), SVAE_DEP8(a, 8) : : "memory");
  asm volatile("" : SVAE_DEP8(b, 0), SVAE_DEP8(b, 8) : : "memory");
}
__device__ __forceinline__ void tmem_wait_ld16(uint32_t (&a)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;" : SVAE_DEP8(a, 0), SVAE_DEP8(a, 8) : : "memory");
}

// ---- descriptors -----------------------------------------------------------------------------------
// UMMA shared-memory matrix descriptor (sm_100): start address, LBO, SBO (all >> 4), version 1, swizzle mode.
//   swizzle_bytes: 128 -> layout_type 2, 64 -> 4, 32 -> 6, 0 -> none.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes, int swizzle_bytes) {
  uint64_t layout = swizzle_bytes == 128 ? 2 : swizzle_bytes == 64 ? 4 : swizzle_bytes == 32 ? 6 : 0;
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;       // descriptor version (Blackwell)
  d |= layout << 61;
  return d;
}

// kind::f16 instruction descriptor: fp32 accumulate, A/B both `fmt` (0 = f16, 1 = bf16), majors 0 = K, 1 = MN.
__host__ __device__ constexpr uint32_t make_idesc(int m, int n, int fmt, int a_major, int b_major) {
  return (1u << 4) | ((uint32_t)fmt << 7) | ((uint32_t)fmt << 10) | ((uint32_t)a_major << 15) | ((uint32_t)b_major << 16) |
         ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// Ties the registers of a preceding tcgen05.ld to the wait, so no use of them can be scheduled above it.
__device__ __forceinline__ void tmem_wait_ld(uint32_t (&r)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;" : SVAE_DEP8(r, 0), SVAE_DEP8(r, 8) : : "memory");
  asm volatile("" : SVAE_DEP8(r, 16), SVAE_DEP8(r, 24) : : "memory");
}
__device__ __forceinline__ void tmem_wait_ld(uint32_t (&a)[32], uint32_t (&b)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;" : SVAE_DEP8(a, 0), SVAE_DEP8(a, 8) : : "memory");
  asm volatile("" : SVAE_DEP8(a, 16), SVAE_DEP8(a, 24) : : "memory");
  asm volatile("" : SVAE_DEP8(b, 0), SVAE_DEP8(b, 8) : : "memory");
  asm volatile("" : SVAE_DEP8(b, 16), SVAE_DEP8(b, 24) : : "memory");
}

__device__ __forceinline__ float fmax3(float a, float b, float c) {
  float r;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}

// barrier among `nthreads` threads of named barrier `id` that also ORs a predicate across them
__device__ __forceinline__ bool bar_red_or(int id, int nthreads, uint32_t pred) {
  uint32_t out;
  asm volatile(
      "{\n\t.reg .pred p, q;\n\tsetp.ne.u32 p, %3, 0;\n\tbar.red.or.pred q, %1, %2, p;\n\tselp.u32 %0, 1, 0, q;\n\t}"
      : "=r"(out)
      : "r"(id), "r"(nthreads), "r"(pred)
      : "memory");
  return out != 0;
}

// ---- warp-convergent issue ---------------------------------------------------------------------------------
// The `_w` wrappers are executed by ALL 32 lanes of a warp with warp-uniform operands; one lane is elected inside
// the asm.  Issuing from an `if (lane == 0)` branch instead makes ptxas treat every operand as divergent and wrap
// each UTCHMMA / UTMALDG in an ELECT + R2UR waterfall loop: measured 127 cycles per tcgen05.mma versus 75 here
// (profiles/README.md).
__device__ __forceinline__ int warp_index() { return __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0); }

__device__ __forceinline__ void mma_ss_w(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, e;\n\telect.sync _|e, 0xffffffff;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void mma_ts_w(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, e;\n\telect.sync _|e, 0xffffffff;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tc_commit_w(uint64_t* bar) {
  asm volatile(
      "{\n\t.reg .pred e;\n\telect.sync _|e, 0xffffffff;\n\t"
      "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx_w(uint64_t* bar, uint32_t bytes) {
  asm volatile(
      "{\n\t.reg .pred e;\n\telect.sync _|e, 0xffffffff;\n\t"
      "@e mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n\t}" ::"r"(smem_u32(bar)), "r"(bytes)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d_w(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2,
                                              int c3) {
  asm volatile(
      "{\n\t.reg .pred e;\n\telect.sync _|e, 0xffffffff;\n\t"
      "@e cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];\n\t}"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

__device__ __forceinline__ void tma_load_2d_w(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "{\n\t.reg .pred e;\n\telect.sync _|e, 0xffffffff;\n\t"
      "@e cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n\t}"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}

// Dependency helpers for batched tcgen05.ld: after ONE wait, tie further register arrays to it.
__device__ __forceinline__ void tmem_dep(uint32_t (&r)[32]) {
  asm volatile("" : SVAE_DEP8(r, 0), SVAE_DEP8(r, 8) : : "memory");
  asm volatile("" : SVAE_DEP8(r, 16), SVAE_DEP8(r, 24) : : "memory");
}

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void named_bar_arrive(int id, int nthreads) {
  asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

}  // namespace ptx
}  // namespace svae
