// Shared device helpers: Philox4x32-10, bit->float maps, vector access, TMA bulk copies.
// The RNG stream layout is specified (and restated in numpy for the tests) in oracle/philox.py.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace mpe {

constexpr int kWarp = 32;

// ----------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al., SC'11).  counter = (gid_lo, gid_hi, t, domain<<16 | slot).
// ----------------------------------------------------------------------------------------------
enum : uint32_t { kDomainReset = 1, kDomainGoal = 2, kDomainGumbel = 3, kDomainRespawn = 4, kDomainReplay = 5 };

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += 0x9E3779B9u;
    k.y += 0xBB67AE85u;
  }
  return c;
}

__device__ __forceinline__ uint4 philox_raw(uint64_t seed, uint64_t gid, uint32_t t, uint32_t domain,
                                            uint32_t slot) {
  return philox4x32_10(make_uint4((uint32_t)gid, (uint32_t)(gid >> 32), t, (domain << 16) | slot),
                       make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
}

// U[-1, 1): a 24-bit integer scaled by 2^-23, exact in fp32 and fp64.
template <typename T>
__device__ __forceinline__ T bits_to_pos(uint32_t r) {
  return (T)(r >> 8) * (T)1.1920928955078125e-07 - (T)1;
}

// NC independent Philox4x32-10 blocks under one key, advanced round by round: the compiler keeps the source order,
// so this is what gives the integer pipe NC independent multiply chains instead of one after the other.
template <int NC>
__device__ __forceinline__ void philox4x32_10_batch(uint4 (&c)[NC], uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
#pragma unroll
    for (int i = 0; i < NC; ++i) {
      const uint32_t hi0 = __umulhi(0xD2511F53u, c[i].x), lo0 = 0xD2511F53u * c[i].x;
      const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[i].z), lo1 = 0xCD9E8D57u * c[i].z;
      c[i] = make_uint4(hi1 ^ c[i].y ^ k.x, lo1, hi0 ^ c[i].w ^ k.y, lo0);
    }
    k.x += 0x9E3779B9u;
    k.y += 0xBB67AE85u;
  }
}
__device__ __forceinline__ uint4 philox_counter(uint64_t gid, uint32_t t, uint32_t domain, uint32_t slot) {
  return make_uint4((uint32_t)gid, (uint32_t)(gid >> 32), t, (domain << 16) | slot);
}
__device__ __forceinline__ uint2 philox_key(uint64_t seed) { return make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)); }

// Gumbel(0,1) from raw bits, NV values in lock-step: u = ((r >> 9) + 0.5) * 2^-23 in (0,1), exact in fp32;
// g = -log(-log(u)).  The inner log must be accurate (the outer log turns its RELATIVE error into absolute error of
// g): branch-free Cephes logf - mantissa folded into [sqrt(1/2), sqrt(2)), degree-8 polynomial, ln2 split hi/lo -
// max relative error 8e-8 over all 2^23 possible u (checked exhaustively on the host); the library logf has
// special-case branches that would put every evaluation into its own basic blocks.  The outer log only needs
// absolute accuracy (~5e-7), which the lg2.approx-based intrinsic gives for E in (6e-8, 17).
// Each stage runs over all NV values before the next stage starts, because ptxas does not interleave independent
// dependency chains by itself (measured: 5 scalar evaluations in a row ran serially, ~150 cycles each).
template <int NV>
__device__ __forceinline__ void bits_to_gumbel_batch(const uint32_t (&r)[NV], float (&g)[NV]) {
  float f[NV], fe[NV], z[NV], p[NV];
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    const float u = ((float)(r[v] >> 9) + 0.5f) * 1.1920928955078125e-07f;
    const int i = __float_as_int(u);
    const int e = (i - 0x3f3504f3) >> 23;
    f[v] = __int_as_float(i - (e << 23)) - 1.0f;
    fe[v] = (float)e;
    z[v] = f[v] * f[v];
    p[v] = 7.0376836292e-2f;
  }
  const float coef[8] = {-1.1514610310e-1f, 1.1676998740e-1f, -1.2420140846e-1f, 1.4249322787e-1f,
                         -1.6668057665e-1f, 2.0000714765e-1f, -2.4999993993e-1f, 3.3333331174e-1f};
#pragma unroll
  for (int j = 0; j < 8; ++j)
#pragma unroll
    for (int v = 0; v < NV; ++v) p[v] = fmaf(p[v], f[v], coef[j]);
#pragma unroll
  for (int v = 0; v < NV; ++v) p[v] = (f[v] * z[v]) * p[v];
#pragma unroll
  for (int v = 0; v < NV; ++v) p[v] = fmaf(fe[v], -2.12194440e-4f, p[v]);
#pragma unroll
  for (int v = 0; v < NV; ++v) p[v] = fmaf(-0.5f, z[v], p[v]);
#pragma unroll
  for (int v = 0; v < NV; ++v) p[v] = fmaf(fe[v], 0.693359375f, f[v] + p[v]);
#pragma unroll
  for (int v = 0; v < NV; ++v) g[v] = -__logf(-p[v]);
}
__device__ __forceinline__ float bits_to_gumbel(uint32_t r) {
  const uint32_t rr[1] = {r};
  float g[1];
  bits_to_gumbel_batch<1>(rr, g);
  return g[0];
}

// ----------------------------------------------------------------------------------------------
// real-type traits: float state is {px,py,vx,vy} float4 / {x,y} float2; double uses 2x double2.
// ----------------------------------------------------------------------------------------------
template <typename T>
struct Vec4 {
  T x, y, z, w;
};
template <typename T>
struct Vec2 {
  T x, y;
};

__device__ __forceinline__ Vec4<float> ld4(const float *p) {
  const float4 v = *reinterpret_cast<const float4 *>(p);
  return {v.x, v.y, v.z, v.w};
}
__device__ __forceinline__ Vec4<double> ld4(const double *p) {
  const double2 a = *reinterpret_cast<const double2 *>(p);
  const double2 b = *reinterpret_cast<const double2 *>(p + 2);
  return {a.x, a.y, b.x, b.y};
}
__device__ __forceinline__ void st4(float *p, Vec4<float> v) {
  *reinterpret_cast<float4 *>(p) = make_float4(v.x, v.y, v.z, v.w);
}
__device__ __forceinline__ void st4(double *p, Vec4<double> v) {
  *reinterpret_cast<double2 *>(p) = make_double2(v.x, v.y);
  *reinterpret_cast<double2 *>(p + 2) = make_double2(v.z, v.w);
}
__device__ __forceinline__ Vec2<float> ld2(const float *p) {
  const float2 v = *reinterpret_cast<const float2 *>(p);
  return {v.x, v.y};
}
__device__ __forceinline__ Vec2<double> ld2(const double *p) {
  const double2 v = *reinterpret_cast<const double2 *>(p);
  return {v.x, v.y};
}
__device__ __forceinline__ void st2(float *p, Vec2<float> v) {
  *reinterpret_cast<float2 *>(p) = make_float2(v.x, v.y);
}
__device__ __forceinline__ void st2(double *p, Vec2<double> v) {
  *reinterpret_cast<double2 *>(p) = make_double2(v.x, v.y);
}

// ----------------------------------------------------------------------------------------------
// TMA bulk copies (cp.async.bulk, SASS UBLKCP) + mbarrier helpers.  Sizes/addresses 16 B aligned.
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}

__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// shared -> global, completion tracked by the issuing thread's bulk async-group
__device__ __forceinline__ void bulk_store(void *gdst, const void *ssrc, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst),
               "r"(smem_u32(ssrc)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// wait until the smem SOURCE of all committed bulk stores has been read (smem reusable)
__device__ __forceinline__ void bulk_wait_read_all() {
  asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
// ... of all but the most recent committed group (double-buffered staging)
__device__ __forceinline__ void bulk_wait_read_1() {
  asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
}

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  // try_wait suspends the thread in hardware until the phase completes or the time hint (ns) expires, so a
  // waiting warp does not burn issue slots of the SM sub-partition it shares with working warps
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t"
      "}" ::"r"(smem_u32(bar)),
      "r"(parity), "r"(1000000u)
      : "memory");
}
// global -> shared, completes on an mbarrier (complete_tx)
__device__ __forceinline__ void bulk_load(void *sdst, const void *gsrc, uint32_t bytes, uint64_t *bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(sdst)),
      "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

}  // namespace mpe
