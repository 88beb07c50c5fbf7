// tcgen05 / TMEM building blocks (sm_100a inline PTX) for the tensor-core actor path.
//
// Operand convention used everywhere in this repo (K-major, no swizzle, "interleave" canonical layout):
//   an operand of `rows` x K 16-bit elements lives in shared memory as [K/8][rows][8] - the 8
//   K-consecutive elements of one row are one 16 B vector, the vectors of consecutive rows are
//   contiguous.  A core matrix (8 rows x 16 B) is therefore 128 contiguous bytes;
//   SBO (next 8-row group) = 128 B, LBO (next K-chunk of 8) = rows * 16 B.
//   One kind::f16 MMA consumes K = 16 = two K-chunks starting at the descriptor's start address.
// Accumulators (M = 128, cta_group::1): D[row][col] at TMEM lane `row`, column `base + col`.
// An A operand in TMEM: lane = row, one 32-bit column holds the two halves k = 2c (low), 2c+1 (high).
#pragma once
#include <cuda_fp16.h>

#include "common.cuh"

namespace mpe {

// Weights are stored as 16 w (kWScale) so that the lo halves of the split stay normal fp16 values; the gate biases
// are stored pre-multiplied by -log2(e) (-2 log2(e) for the cell gate): the argument form of ex2.
constexpr float kWScale = 16.0f, kWInv = 0.0625f, kLog2e = 1.4426950408889634f;

// ---- TMEM allocation (one full warp executes these) ----
__device__ __forceinline__ void tmem_alloc(uint32_t *smem_slot, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_free(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ---- descriptors ----
// 64-bit shared-memory matrix descriptor: start >> 4 | LBO >> 4 << 16 | SBO >> 4 << 32 | version 1 << 46 | no swizzle
__device__ __forceinline__ uint64_t make_smem_desc(const void *smem_ptr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  const uint32_t addr = smem_u32(smem_ptr);
  uint64_t d = 0;
  d |= (uint64_t)((addr & 0x3FFFF) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  return d;
}
// 32-bit instruction descriptor, kind::f16: D = fp32, A = B = fp16, both K-major, dense
__host__ __device__ constexpr uint32_t make_idesc_f16(int M, int N) {
  return (1u << 4) | (0u << 7) | (0u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// ---- MMA issue (ONE thread) ----
__device__ __forceinline__ void mma_f16_ss(uint32_t tmem_d, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                           bool accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"((uint32_t)accumulate)
      : "memory");
}
__device__ __forceinline__ void mma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t b_desc, uint32_t idesc,
                                           bool accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(tmem_d),
      "r"(tmem_a), "l"(b_desc), "r"(idesc), "r"((uint32_t)accumulate)
      : "memory");
}
// all MMAs issued so far by this thread arrive on `bar` when complete (implies fence::before_thread_sync)
__device__ __forceinline__ void mma_commit(uint64_t *bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// ---- TMEM <-> registers, 32 lanes x 32-bit, N consecutive columns; warp w touches lanes 32*(w%4).. ----
#define MPE_R8(v, o) "=r"(v[o + 0]), "=r"(v[o + 1]), "=r"(v[o + 2]), "=r"(v[o + 3]), "=r"(v[o + 4]), "=r"(v[o + 5]), "=r"(v[o + 6]), "=r"(v[o + 7])
#define MPE_W8(v, o) "r"(v[o + 0]), "r"(v[o + 1]), "r"(v[o + 2]), "r"(v[o + 3]), "r"(v[o + 4]), "r"(v[o + 5]), "r"(v[o + 6]), "r"(v[o + 7])

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,"
      "%30,%31}, [%32];"
      : MPE_R8(v, 0), MPE_R8(v, 8), MPE_R8(v, 16), MPE_R8(v, 24)
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : MPE_R8(v, 0), MPE_R8(v, 8)
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&v)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : MPE_R8(v, 0)
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tmem_st4(uint32_t taddr, const uint32_t (&v)[4]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(taddr), "r"(v[0]), "r"(v[1]),
               "r"(v[2]), "r"(v[3])
               : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,"
      "%31,%32};" ::"r"(taddr),
      MPE_W8(v, 0), MPE_W8(v, 8), MPE_W8(v, 16), MPE_W8(v, 24)
      : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(
          taddr),
      MPE_W8(v, 0), MPE_W8(v, 8)
      : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---- fp32 -> (hi, lo) fp16 split: x = hi + lo + O(2^-22 |x|) (absolute floor 2^-25 from fp16 subnormals) ----
__device__ __forceinline__ void split_f16(float x, __half &hi, __half &lo) {
  hi = __float2half_rn(x);
  lo = __float2half_rn(x - __half2float(hi));
}
__device__ __forceinline__ uint32_t pack_h2(__half a, __half b) {
  const __half2 h = __halves2half2(a, b);
  return *reinterpret_cast<const uint32_t *>(&h);
}

}  // namespace mpe
