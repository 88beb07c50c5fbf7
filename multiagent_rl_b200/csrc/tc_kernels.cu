// Tensor-core (tcgen05 / TMEM) version of the actor forward (teams of 2, 3, 4, 6, 8, 9, 12) and of the fused
// rollout step (teams of 2 and 3): one kernel, k_tc2, whose warp roles and TMEM / shared-memory layout are described
// above its definition.
//
// Reference rows: same as actor_kernels.cu (rls/model/ac_network_multi_gumbel.py:52-67,
// rls/agent/multiagent/ddpg_gumbel_fix.py:86-116, experiments/run.py:36-65).
//
// Why tensor cores: ncu on the fp32 SIMT kernel shows DRAM 0.2 %, FMA pipe 54 %, issue 64 % - the batched
// LSTM GEMMs are contraction-bound.  Why fp16 hi/lo: the acting path must reproduce the reference's fp32
// logits to ~1e-6 so that the sampled index is bit-exact under identical noise; every fp32 operand x is
// split as x = hi + lo (two fp16 values, 22 significant bits) and each product is three kind::f16 MMAs
// (hi*hi + lo*hi + hi*lo) accumulated in fp32 in TMEM.  Weights are pre-split (and pre-scaled by 16 so
// that the lo halves stay normal) when they are loaded (pack_kernels.cu); activations are split by the epilogue that produces them.
#include <cuda_fp16.h>

#include <cstdlib>

#include "actor_launch.h"
#include "env_core.cuh"
#include "launch.h"
#include "tc_common.cuh"

namespace mpe {

constexpr int kRows = 128;
constexpr uint32_t kChunkA = kRows * 16;  // bytes of one K-chunk (8 halves) of a 128-row A operand

// ------------------------------------------------------------------------------------------------
// host: layout of the fp16 hi/lo weight image (packed by pack_kernels.cu)
// ------------------------------------------------------------------------------------------------
void tc_layout(int D, int A0, int A1, TcDev *o) {
  o->D = D; o->A0 = A0; o->A1 = A1; o->A = A0 + A1;
  o->Kx = D <= 16 ? 16 : (D <= 32 ? 32 : 0);
  uint32_t off = 0;
  for (int d = 0; d < 2; ++d)
    for (int hl = 0; hl < 2; ++hl) { o->off_wih[d][hl] = off; off += kHid * kGateN * 2; }
  for (int d = 0; d < 2; ++d)
    for (int hl = 0; hl < 2; ++hl) { o->off_whh[d][hl] = off; off += kH * kGateN * 2; }
  for (int hl = 0; hl < 2; ++hl) { o->off_w1[hl] = off; off += (o->Kx > 0 ? o->Kx : 16) * kHid * 2; }
  for (int d = 0; d < 2; ++d)
    for (int hl = 0; hl < 2; ++hl) { o->off_w2[d][hl] = off; off += kW2Bytes; }
  o->off_w2f = off; off += kHid * 16 * 4;  // dense2 heads, fp32 [k = dir*32 + unit][16]
  o->off_bg = off; off += 2 * kGateN * 4;
  o->off_b1 = off; off += kHid * 4;
  o->off_b2 = off; off += 16 * 4;
  o->bytes = (off + 127) / 128 * 128;
}

bool tc_supported(const TcDev &t) { return t.Kx > 0 && t.A <= 16; }

// ------------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------------

__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bar_sync_n(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }

// 8 fp32 values -> one 16 B vector of fp16 hi parts and one of lo parts, stored at the row's slot of a K-chunk
__device__ __forceinline__ void store_chunk_split(unsigned char *hi_chunk, unsigned char *lo_chunk, int row,
                                                  const float (&v)[8]) {
  uint32_t h[4], l[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    __half h0, l0, h1, l1;
    split_f16(v[2 * i], h0, l0);
    split_f16(v[2 * i + 1], h1, l1);
    h[i] = pack_h2(h0, h1);
    l[i] = pack_h2(l0, l1);
  }
  *reinterpret_cast<uint4 *>(hi_chunk + row * 16) = make_uint4(h[0], h[1], h[2], h[3]);
  *reinterpret_cast<uint4 *>(lo_chunk + row * 16) = make_uint4(l[0], l[1], l[2], l[3]);
}

// three-term split product D (+)= A*B with A and B in shared memory, K = 16 * kblocks
__device__ __forceinline__ void mma3_ss(uint32_t tmem_d, const unsigned char *a_hi, const unsigned char *a_lo,
                                        uint32_t a_lbo, const unsigned char *b_hi, const unsigned char *b_lo,
                                        uint32_t b_lbo, int kblocks, uint32_t idesc, bool accumulate) {
  for (int kb = 0; kb < kblocks; ++kb) {
    const uint64_t ah = make_smem_desc(a_hi + kb * 2 * a_lbo, a_lbo, 128), al = make_smem_desc(a_lo + kb * 2 * a_lbo, a_lbo, 128);
    const uint64_t bh = make_smem_desc(b_hi + kb * 2 * b_lbo, b_lbo, 128), bl = make_smem_desc(b_lo + kb * 2 * b_lbo, b_lbo, 128);
    mma_f16_ss(tmem_d, ah, bh, idesc, accumulate || kb > 0);
    mma_f16_ss(tmem_d, al, bh, idesc, true);
    mma_f16_ss(tmem_d, ah, bl, idesc, true);
  }
}
// same with the A operand in TMEM (hi at column a_hi, lo at column a_lo; 8 columns per K = 16 block)
__device__ __forceinline__ void mma3_ts(uint32_t tmem_d, uint32_t a_hi, uint32_t a_lo, const unsigned char *b_hi,
                                        const unsigned char *b_lo, uint32_t b_lbo, int kblocks, uint32_t idesc,
                                        bool accumulate) {
  for (int kb = 0; kb < kblocks; ++kb) {
    const uint64_t bh = make_smem_desc(b_hi + kb * 2 * b_lbo, b_lbo, 128), bl = make_smem_desc(b_lo + kb * 2 * b_lbo, b_lbo, 128);
    mma_f16_ts(tmem_d, a_hi + kb * 8, bh, idesc, accumulate || kb > 0);
    mma_f16_ts(tmem_d, a_lo + kb * 8, bh, idesc, true);
    mma_f16_ts(tmem_d, a_hi + kb * 8, bl, idesc, true);
  }
}

// Optional phase timeline (MPE_TC_TIMELINE=1): clock64 stamps of the first tile of every warpgroup, read back
// with the (undeclared, debug-only) export mpe_debug_tc_timeline.
__device__ unsigned long long g_tc_timeline[148 * 128];
#ifdef MPE_TC_PHASES  // instrumented build only (python -m multiagent_rl_b200.build --variant phases MPE_TC_PHASES)
#define TL(role, i)                                                                                              \
  do {                                                                                                           \
    if (dbg && first_tile && blockIdx.x < 148) g_tc_timeline[blockIdx.x * 128 + (role) * 32 + (i)] = clock64(); \
  } while (0)
#else
#define TL(role, i)
#endif

// barriers of one warpgroup's pipeline (indices into its own block of the barrier array); B_L: the tile's dense2
// logits are complete in TMEM (heads on the tensor pipe only)
enum { B_X = 0, B_D1, B_H1, B_G, B_H, B_L, B_PER_WG };

// operand buffers: all agents resident (N <= 3); a ring of 4 (teams of 4 / 6: 16-wide operands, shared memory to
// spare) or 2 (9 / 12 agents: 32-wide operands) buffers refilled ahead of the dense1 GEMMs
__host__ __device__ constexpr int tc_x_slots(int N) { return N <= 3 ? N : (N <= 6 ? 4 : 2); }
__host__ __device__ inline size_t tc_x_bytes(int N, int Kx) { return (size_t)tc_x_slots(N) * 2 * (Kx / 8) * kChunkA; }

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// exp(-x) with the exponent clamped so that products of two such terms stay finite
__device__ __forceinline__ float exp_neg(float x) { return ex2_approx(fminf(-1.4426950408889634f * x, 57.0f)); }

// dense1 epilogue for 32 hidden units of one env row: h1 = relu(D1/16 + b1) -> fp16 hi/lo, 16 packed columns each
__device__ __forceinline__ void dense1_half(const uint32_t (&v)[32], const float *b1, uint32_t taddr_hi,
                                            uint32_t lo_off = 32) {
  uint32_t hi[16], lo[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    const float2 bj = *reinterpret_cast<const float2 *>(b1 + 2 * j);
    const float a0 = fmaxf(fmaf(__uint_as_float(v[2 * j]), kWInv, bj.x), 0.0f);
    const float a1 = fmaxf(fmaf(__uint_as_float(v[2 * j + 1]), kWInv, bj.y), 0.0f);
    __half h0, l0, h1, l1;
    split_f16(a0, h0, l0);
    split_f16(a1, h1, l1);
    hi[j] = pack_h2(h0, h1);
    lo[j] = pack_h2(l0, l1);
  }
  tmem_st16(taddr_hi, hi);
  tmem_st16(taddr_hi + lo_off, lo);
}

// ---- packed fp32x2 arithmetic (sm_100 FFMA2 / FADD2 / FMUL2): one issue slot for two lanes of cell math ----
typedef unsigned long long f2;
__device__ __forceinline__ f2 pk(float lo, float hi) { f2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ f2 pk(uint32_t lo, uint32_t hi) { f2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(lo), "r"(hi)); return r; }
__device__ __forceinline__ void upk(f2 v, float &lo, float &hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f2 fma2(f2 a, f2 b, f2 c) { f2 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
__device__ __forceinline__ f2 add2(f2 a, f2 b) { f2 d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ f2 mul2(f2 a, f2 b) { f2 d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ float rcp_approx(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

// reciprocal of d >= 1 on the FMA pipe (no MUFU): bit-trick seed (<= 12 % off) + 3 Newton steps (-> ~4e-8), packed
__device__ __forceinline__ f2 rcp2_newton(f2 d) {
  float d0, d1;
  upk(d, d0, d1);
  f2 r = pk(__uint_as_float(0x7EF311C7u - __float_as_uint(d0)), __uint_as_float(0x7EF311C7u - __float_as_uint(d1)));
  const f2 nd = mul2(d, pk(-1.0f, -1.0f)), TWO = pk(2.0f, 2.0f);
#pragma unroll
  for (int it = 0; it < 3; ++it) r = mul2(r, fma2(nd, r, TWO));
  return r;
}

// LSTM cell math for 8 units of one env row.  v = 32 gate accumulator columns (scaled by 16) in the packed order
// [i_a i_b f_a f_b g_a g_b o_a o_b] per pair of units (a, b) = (2p, 2p+1), so that the two cells of a pair sit in
// adjacent registers and every FP32 operation of the cell is one FFMA2/FADD2/FMUL2.  bg = 32 biases in the same
// order, pre-multiplied by -log2(e) (x2 for the g gate); c = the 4 packed cell-state pairs.  The MUFU pipe is the
// floor of this kernel, so the cell is arranged to need 5 MUFU ops (the five ex2) instead of the textbook 10: with
// e* = exp(-x) (arguments clamped so that no product overflows)
//   c' = sigmoid(f) c + sigmoid(i) tanh(g) = [c (1+ei)(1+eg) + (1-eg)(1+ef)] / [(1+ef)(1+ei)(1+eg)]   one reciprocal
//   h  = sigmoid(o) tanh(c') = (1 - ec) / ((1+eo)(1+ec))                                              one reciprocal
// and both reciprocals (denominators >= 1) by a bit-trick seed + 3 Newton steps on the FMA pipe.
__device__ __forceinline__ void lstm_h8(const uint32_t (&v)[32], const float *bg, f2 (&c)[4], float (&hv)[8]) {
  const f2 ONE = pk(1.0f, 1.0f), NEG1 = pk(-1.0f, -1.0f);
  const f2 S1 = pk(-kWInv * kLog2e, -kWInv * kLog2e), S2 = pk(-2.0f * kWInv * kLog2e, -2.0f * kWInv * kLog2e);
  const f2 S3 = pk(-2.0f * kLog2e, -2.0f * kLog2e);
  constexpr float kClamp = 40.0f;  // e <= 2^40: sigmoid floors at 9e-13, tanh saturates to 1 - 2e-12
  f2 pO[4];
  // stage 1: exponentials of the four gates, then the new cell state with a single reciprocal
#pragma unroll
  for (int p = 0; p < 4; ++p) {
    const ulonglong2 b0 = *reinterpret_cast<const ulonglong2 *>(bg + p * 8);      // (b_i pair, b_f pair)
    const ulonglong2 b1 = *reinterpret_cast<const ulonglong2 *>(bg + p * 8 + 4);  // (b_g pair, b_o pair)
    const f2 aI = fma2(pk(v[8 * p + 0], v[8 * p + 1]), S1, b0.x), aF = fma2(pk(v[8 * p + 2], v[8 * p + 3]), S1, b0.y);
    const f2 aG = fma2(pk(v[8 * p + 4], v[8 * p + 5]), S2, b1.x), aO = fma2(pk(v[8 * p + 6], v[8 * p + 7]), S1, b1.y);
    float x0, x1;
    upk(aI, x0, x1); const f2 eI = pk(ex2_approx(fminf(x0, kClamp)), ex2_approx(fminf(x1, kClamp)));
    upk(aF, x0, x1); const f2 eF = pk(ex2_approx(fminf(x0, kClamp)), ex2_approx(fminf(x1, kClamp)));
    upk(aG, x0, x1); const f2 eG = pk(ex2_approx(fminf(x0, kClamp)), ex2_approx(fminf(x1, kClamp)));
    upk(aO, x0, x1); const f2 eO = pk(ex2_approx(fminf(x0, kClamp)), ex2_approx(fminf(x1, kClamp)));
    const f2 F = add2(eF, ONE), P = mul2(add2(eI, ONE), add2(eG, ONE));
    const f2 num = fma2(c[p], P, mul2(fma2(eG, NEG1, ONE), F));
    c[p] = mul2(num, rcp2_newton(mul2(F, P)));  // den >= 1: Newton on the FMA pipe (measured: -3 % kernel time vs MUFU.RCP)
    pO[p] = add2(eO, ONE);
  }
  // stage 2: h = sigmoid(o) tanh(c) = (1 - ec) / ((1 + eo)(1 + ec)), reciprocal on the FMA pipe
#pragma unroll
  for (int p = 0; p < 4; ++p) {
    float x0, x1;
    upk(mul2(c[p], S3), x0, x1);
    const f2 eC = pk(ex2_approx(fminf(x0, kClamp)), ex2_approx(fminf(x1, kClamp)));
    const f2 r = rcp2_newton(mul2(pO[p], add2(eC, ONE)));
    upk(mul2(fma2(eC, NEG1, ONE), r), hv[2 * p], hv[2 * p + 1]);
  }
}

// The outputs of 8 units' h: h as an fp16 hi/lo K-chunk of the recurrent A operand when `store_h`, relu(h) for the
// dense3 head when `hcat8` is set.
__device__ __forceinline__ void h8_outputs(const float (&hv)[8], unsigned char *h_chunk, int row, bool store_h,
                                           float *hcat8) {
  if (store_h) store_chunk_split(h_chunk, h_chunk + 8192, row, hv);
  if (hcat8 != nullptr) {  // relu(h) of these 8 units for the dense3 head (actor_forward with next_state; 32 B aligned)
    *reinterpret_cast<float4 *>(hcat8) = make_float4(fmaxf(hv[0], 0.0f), fmaxf(hv[1], 0.0f), fmaxf(hv[2], 0.0f), fmaxf(hv[3], 0.0f));
    *reinterpret_cast<float4 *>(hcat8 + 4) = make_float4(fmaxf(hv[4], 0.0f), fmaxf(hv[5], 0.0f), fmaxf(hv[6], 0.0f), fmaxf(hv[7], 0.0f));
  }
}

// Cell math of 8 units with the dense2 heads on the FMA pipe (teams of > 3, two-head actors): pl = packed dense2
// partial sums, FFMA2 over pairs of head entries with the weights broadcast from smem.
template <int APAD>
__device__ __forceinline__ void lstm_chunk(const uint32_t (&v)[32], const float *bg, const float *w2rows, f2 (&c)[4],
                                           f2 (&pl)[APAD / 2], unsigned char *h_chunk, int row, bool store_h,
                                           float *hcat8 = nullptr) {
  float hv[8];
  lstm_h8(v, bg, c, hv);
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float rj = fmaxf(hv[j], 0.0f);
    const f2 rr = pk(rj, rj);
#pragma unroll
    for (int a = 0; a < APAD; a += 4) {
      const ulonglong2 wv = *reinterpret_cast<const ulonglong2 *>(w2rows + j * 16 + a);
      pl[a / 2] = fma2(rr, wv.x, pl[a / 2]);
      pl[a / 2 + 1] = fma2(rr, wv.y, pl[a / 2 + 1]);
    }
  }
  h8_outputs(hv, h_chunk, row, store_h, hcat8);
}

// Cell math of 8 units with the dense2 heads on the tensor pipe (teams of <= 3 with one head): relu(h) as fp16 hi/lo
// pairs into the tile's dense2 A operand in TMEM (4 hi columns at taddr, the lo columns 16 further), read by the
// issuer's dense2 MMAs once the cell is complete.
__device__ __forceinline__ void lstm_chunk_tc(const uint32_t (&v)[32], const float *bg, f2 (&c)[4], uint32_t taddr,
                                              unsigned char *h_chunk, int row, bool store_h, float *hcat8) {
  float hv[8];
  lstm_h8(v, bg, c, hv);
  uint32_t hi[4], lo[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    __half h0, l0, h1, l1;
    split_f16(fmaxf(hv[2 * i], 0.0f), h0, l0);
    split_f16(fmaxf(hv[2 * i + 1], 0.0f), h1, l1);
    hi[i] = pack_h2(h0, h1);
    lo[i] = pack_h2(l0, l1);
  }
  tmem_st4(taddr, hi);
  tmem_st4(taddr + 16, lo);
  h8_outputs(hv, h_chunk, row, store_h, hcat8);
}

// ------------------------------------------------------------------------------------------------
// k_tc2: one persistent CTA per SM walks pairs of tiles (tile = 128 envs = 128 TMEM lanes).  Warps 0-7 are two
// epilogue warpgroups, warp 8 / 9 issues the tcgen05.mma stream of tile 0 / 1, and for teams of > 3 agents warps
// 10 / 11 are the operand warps described in the kernel.  BOTH warpgroups work on EVERY cell - warpgroup h
// takes hidden units 16h..16h+15 of the cell (and 32 of the 64 dense1 columns), and the cells of the two tiles are
// interleaved in one software pipeline:
//      E1(A,k)  C(B,k-1)  E1(B,k)  C(A,k)  E1(A,k+1)  C(B,k) ...
// (E1 = dense1 epilogue -> h1 operand in TMEM, C = LSTM cell math on the gate accumulators).  While all eight warps
// run the cell math of one tile, the tensor pipe runs the gate GEMM of the other, so no warp ever waits for an MMA
// in steady state and every SM sub-partition always has two warps in the same MUFU-heavy phase.
// Warpgroup h owns tile h for everything that is per env (obs operands, sampling, World.step, outputs).  Teams of
// <= 3 with one head of <= 8 entries run the dense2 heads on the tensor pipe: every cell writes relu(h) into a TMEM
// A operand and the issuer accumulates [128 x 32] x [32 x 16] per cell into the agent's logit columns, which the
// owner reads after the pipeline.  Large teams and two-head actors keep FFMA2 heads whose per-cell shares travel
// through global scratch rows (their TMEM has no room for the logit columns / the heads are 16 entries wide).
// ------------------------------------------------------------------------------------------------
__host__ __device__ constexpr bool tc2_tc_heads(int N, int APAD) { return N <= 3 && APAD <= 8; }
// TMEM columns of a tile with the heads on the tensor pipe: logits of agent t at kLogitCol + 8t (one M = 128, N = 16
// accumulator per pair of agents), the relu(h) A operand (K = 32: 16 hi columns, then 16 lo columns) at kReluCol
constexpr uint32_t kLogitCol = 192, kReluCol = 224;
__host__ __device__ inline size_t tc2_tile_bytes(int N, int Kx) {
  // obs operands, recurrent h operand, action bytes
  return tc_x_bytes(N, Kx) + 16384 + (size_t)((kRows * N * 2 + 127) / 128 * 128);
}
// per tile: operand ring buffer q (< 4) ready / free again.  B2_OBS has no waiter; it stays (with its mbar_init)
// because without it ptxas reschedules the large-team kernels, a change that wants its own measurement.
enum { B2_XR = 0, B2_XF = 4, B2_OBS = 8, B2_EXTRA = 9 };
__host__ __device__ inline size_t tc2_smem_bytes(uint32_t wbytes, int N, int Kx) {
  return (size_t)wbytes + 2 * tc2_tile_bytes(N, Kx) + (1 + 2 * B_PER_WG + 2 * B2_EXTRA) * 8 + 64;
}
// dense2 shares of large teams: [CTA][tile 0/1][warpgroup half][cell 0..2N-1][APAD/2 packed pairs][128 rows] f2
__host__ __device__ inline size_t tc2_scratch_f2_per_cta(int N, int APAD) { return (size_t)2 * 2 * 2 * N * (APAD / 2) * kRows; }
__host__ __device__ constexpr int tc2_threads(int N) { return N > 3 ? 384 : 320; }  // + two service warps for large teams

// INFO (fused rollouts only): also write the benchmark_data of every env-step to ro.info_i / ro.info_f.  A template
// flag rather than a test of the pointers, so that the kernel of a rollout without them stays the same code.
template <int SC, int N, bool FUSED, int APAD, bool INFO = false>
__global__ void __launch_bounds__(tc2_threads(N), 1)
    k_tc2(EnvState<float> s, TcDev w, ActorIO io, RolloutIO ro, int max_episode_len, int64_t ntiles, int dbg) {
  // Large teams (N > 3, actor only): the obs operands do not fit next to the weights, so a per-tile OPERAND WARP
  // (warps 10 / 11; the register file is allocated for 12 warps anyway) streams them from the caller's tensor into a
  // operand ring (4 buffers for 4 / 6 agents, 2 for 9 / 12) ahead of the dense1 GEMMs, and every cell's dense2 share goes to its own
  // global scratch row (L2 resident) from which the owner warpgroup completes the logits and samples after the
  // pipeline.  Inside the pipeline the eight epilogue warps do nothing but the dense1 epilogue and the cell math.
  // (Measured alternatives: refilling from the epilogue warps - 400 B of spills and exposed load latency, slower than
  // the earlier two-pipeline kernel; a service warp that also samples one cell behind the pipeline - its ~11 k
  // instructions per tile slow the two sub-partitions it shares and with them the whole barrier-coupled pipeline.)
  constexpr bool kJit = N > 3;
  // two-head actors of small teams (simple_reference, A = 5 + 10) keep the FFMA heads too: the OTHER warpgroup's
  // shares travel through the scratch rows (the own shares stay in registers)
  constexpr bool kXs = !kJit && APAD > 8;
  // every other small team (one head of <= 8 entries): the heads on the tensor pipe, logits accumulated in TMEM
  constexpr bool kTcHeads = tc2_tc_heads(N, APAD);
  static_assert(!(kJit && FUSED), "the fused rollout keeps every agent of an env in one thread: N <= 3");
  static_assert(FUSED || !INFO, "benchmark_data is a rollout output");
  extern __shared__ __align__(128) unsigned char smem[];
#ifdef MPE_TC_PHASES
  if (dbg && threadIdx.x == 0 && blockIdx.x < 148) {
    unsigned long long gt;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
    g_tc_timeline[blockIdx.x * 128 + 64] = gt;
    g_tc_timeline[blockIdx.x * 128 + 66] = clock64();
  }
#endif
  using Dm = Dims<SC, N>;
  const int D = FUSED ? Dm::D : w.D;
  const int R = N * D;
  const int Kx = w.Kx;
  const int tid = threadIdx.x, warp = tid >> 5;
  const size_t xb = tc_x_bytes(N, Kx);
  const size_t tile_bytes = tc2_tile_bytes(N, Kx);
  unsigned char *sm_w = smem;
  uint64_t *bars = reinterpret_cast<uint64_t *>(smem + w.bytes + 2 * tile_bytes);  // [0] = weights, then 2 x B_PER_WG
  uint64_t *xbars = bars + 1 + 2 * B_PER_WG;  // [tile][B2_XR + buf | B2_XF + buf]
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(xbars + 2 * B2_EXTRA);
  auto tile_smem = [&](int X) { return smem + w.bytes + X * tile_bytes; };

  if (tid == 0) {
    mbar_init(&bars[0], 1);
    for (int g = 0; g < 2; ++g) {
      uint64_t *bb = bars + 1 + g * B_PER_WG;
      mbar_init(&bb[B_X], 128);   // the owner warpgroup wrote the tile's obs operands
      mbar_init(&bb[B_D1], 1);
      mbar_init(&bb[B_H1], 256);  // both warpgroups converted their half of h1
      mbar_init(&bb[B_G], 1);
      mbar_init(&bb[B_H], 256);   // both warpgroups finished their half of the cell
      mbar_init(&bb[B_L], 1);
      for (int q = 0; q < 4; ++q) {
        mbar_init(&xbars[g * B2_EXTRA + B2_XR + q], 32);  // the service warp filled operand buffer q
        mbar_init(&xbars[g * B2_EXTRA + B2_XF + q], 1);   // the dense1 GEMM reading buffer q has completed
      }
      mbar_init(&xbars[g * B2_EXTRA + B2_OBS], 128);      // no waiter, see B2_OBS
    }
    mbar_fence_init();
    mbar_expect_tx(&bars[0], w.bytes);
    bulk_load(sm_w, w.blob, w.bytes, &bars[0]);
  }
  if (warp == 8) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int T = FUSED ? ro.T : 1;
  // TMEM columns of a tile: gate accumulators [0,128) and 64-column h1 slots from 128 on.  A slot first receives the
  // dense1 accumulators of an agent and is then converted IN PLACE into that agent's h1 operand (thread half h owns
  // columns [32h, 32h+32) of the slot: fp16 hi pairs in the first 16, lo pairs in the last 16).  With the heads on
  // the FMA pipe there are two slots (128 / 192) and agent t lives in slot t & 1, so the backward pass finds the h1 of
  // agents N-1 and N-2 still resident: 4 dense1 GEMMs + epilogues per 3-agent tile instead of 6.  With the heads on
  // the tensor pipe [192, 256) holds the logits and the relu(h) operand, one slot remains, and the backward pass
  // recomputes every agent but N-1: 5 dense1 GEMMs + epilogues per 3-agent tile, 3 per 2-agent tile.
  constexpr int kSlots = kTcHeads ? 1 : 2;
  auto agent_of = [](int k) { return k < N ? k : 2 * N - 1 - k; };
  auto need_e1 = [&](int k) { return k < N || agent_of(k) + kSlots < N; };
  auto slot_col = [](int t) { return 128u + 64u * (uint32_t)(t % kSlots); };
  const int64_t npairs = (ntiles + 1) / 2;
  // large teams: index of cell j in the sequence of cells that have a dense1 GEMM (the two resident backward cells
  // N, N+1 are skipped); the operand ring buffer of that GEMM is (index mod ring depth)
  auto d1_index = [](int j) { return j < N ? j : j - 2; };
  constexpr int kRing = kJit ? tc_x_slots(N) : 1;  // power of two

  if (kJit && warp >= 10) {
    // =============================== operand warp of tile X = warp - 10 (large teams) ===============================
    // obs[b][t][:] of the caller's tensor -> fp16 hi/lo ring buffers, in GEMM order, one or two cells ahead of the
    // dense1 GEMMs.  Lane l serves rows l, l+32, l+64, l+96; ring buffer q is reused once the dense1 GEMM that read
    // it has completed (B2_XF, tcgen05.commit).
    const int X = warp - 10, lane = tid & 31;
    unsigned char *sm_x = tile_smem(X);
    uint64_t *xb2 = xbars + X * B2_EXTRA;
    uint32_t ph_xf = 0, filled = 0;  // bit q: phase parity of / first fill done for ring buffer q
    const bool vec2 = (reinterpret_cast<uintptr_t>(io.obs) & 7) == 0 && (D & 1) == 0;
    for (int64_t pair = blockIdx.x; pair < npairs; pair += gridDim.x) {
      const int64_t tile = pair * 2 + X, env0 = tile * kRows;
      const int valid = tile < ntiles ? (int)((io.B - env0) < kRows ? (io.B - env0) : kRows) : 0;
#pragma unroll 1
      for (int j = 0; j < 2 * N; ++j) {
        if (!need_e1(j)) continue;
        const int t = agent_of(j), q = d1_index(j) & (kRing - 1);
        if ((filled >> q) & 1u) { mbar_wait(&xb2[B2_XF + q], (ph_xf >> q) & 1u); ph_xf ^= 1u << q; }
        filled |= 1u << q;
        unsigned char *xh = sm_x + (size_t)(q * 2) * (Kx / 8) * kChunkA, *xl = xh + (size_t)(Kx / 8) * kChunkA;
#pragma unroll 1
        for (int rp = 0; rp < 2; ++rp) {  // two rows per round: 2 x 32 values in registers, loads of both in flight
          float xr[2][32];
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const int r = lane + 32 * (2 * rp + u);
#pragma unroll
            for (int k = 0; k < 32; ++k) xr[u][k] = 0.0f;
            if (r < valid) {
              const float *src = io.obs + (env0 + r) * R + t * D;
              if (vec2) {
#pragma unroll
                for (int k = 0; k < 16; ++k)
                  if (2 * k < D) {
                    const float2 v = *reinterpret_cast<const float2 *>(src + 2 * k);
                    xr[u][2 * k] = v.x; xr[u][2 * k + 1] = v.y;
                  }
              } else {
#pragma unroll
                for (int k = 0; k < 32; ++k)
                  if (k < D) xr[u][k] = src[k];
              }
            }
          }
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const int r = lane + 32 * (2 * rp + u);
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              if (c * 8 < Kx) {
                const float v[8] = {xr[u][c * 8], xr[u][c * 8 + 1], xr[u][c * 8 + 2], xr[u][c * 8 + 3],
                                    xr[u][c * 8 + 4], xr[u][c * 8 + 5], xr[u][c * 8 + 6], xr[u][c * 8 + 7]};
                store_chunk_split(xh + c * kChunkA, xl + c * kChunkA, r, v);
              }
            }
          }
        }
        fence_proxy_async_smem();
        mbar_arrive(&xb2[B2_XR + q]);
      }
    }
  } else if (warp >= 8) {
    // =============================== MMA issuer of tile X = warp - 8 ===============================
    const int X = warp - 8;
    if ((tid & 31) == 0) {
      unsigned char *sm_x = tile_smem(X), *sm_h = sm_x + xb;
      uint64_t *bb = bars + 1 + X * B_PER_WG;
      const uint32_t tmem = tmem_base + X * 256;
      uint32_t ph_x = 0, ph_h1 = 0, ph_h = 0, ph_xr = 0;  // ph_xr: bit q = phase parity of ring buffer q
      uint64_t *xb2 = xbars + X * B2_EXTRA;
      const uint32_t id_g = make_idesc_f16(128, 128), id_d1 = make_idesc_f16(128, 64), id_l = make_idesc_f16(128, 16);
      mbar_wait(&bars[0], 0);
      for (int64_t pair = blockIdx.x; pair < npairs; pair += gridDim.x) {
        for (int it = 0; it < T; ++it) {
          if constexpr (!kJit) {
            mbar_wait(&bb[B_X], ph_x); ph_x ^= 1;
            tc_fence_after();
          }
          // dense1 GEMM of cell j -> the agent's h1 slot.  Small teams: operand buffer = agent (all resident).
          // Large teams: ring buffer (dense1 index mod depth), filled by the operand warp; its completion frees the buffer.
          auto dense1_cell = [&](int j) {
            const int t = agent_of(j), q = d1_index(j) & (kRing - 1), xs = kJit ? q : t;
            if constexpr (kJit) {
              mbar_wait(&xb2[B2_XR + q], (ph_xr >> q) & 1u); ph_xr ^= 1u << q;
              tc_fence_after();
            }
            const unsigned char *xh = sm_x + (size_t)(xs * 2) * (Kx / 8) * kChunkA, *xl = xh + (size_t)(Kx / 8) * kChunkA;
            mma3_ss(tmem + slot_col(t), xh, xl, kChunkA, sm_w + w.off_w1[0], sm_w + w.off_w1[1], kHid * 16, Kx / 16, id_d1, false);
            mma_commit(&bb[B_D1]);
            if constexpr (kJit) mma_commit(&xb2[B2_XF + q]);
          };
          // dense2 heads of cell j, once both warpgroups have written its relu(h): agent t accumulates into columns
          // 8t..8t+7 of its pair's N = 16 accumulator (B operand starting at row 8 for even agents, row 0 for odd ones,
          // the other 8 columns are zero weights).  An even agent's forward cell starts the pair's sums.  Issued
          // before the tile's next gate GEMM, whose B_G commit the next cell's math (which rewrites relu(h)) waits on.
          auto dense2_cell = [&](int j) {
            const int t = agent_of(j), d = j >= N ? 1 : 0;
            const uint32_t boff = (t & 1) ? 0u : 128u;
            const unsigned char *w2_hi = sm_w + (d ? w.off_w2[1][0] : w.off_w2[0][0]) + boff;
            const unsigned char *w2_lo = sm_w + (d ? w.off_w2[1][1] : w.off_w2[0][1]) + boff;
            mma3_ts(tmem + kLogitCol + 16u * (uint32_t)(t >> 1), tmem + kReluCol, tmem + kReluCol + 16, w2_hi, w2_lo,
                    kW2Rows * 16, 2, id_l, d == 1 || (t & 1) == 1);
          };
          dense1_cell(0);
          for (int k = 0; k < 2 * N; ++k) {
            const int d = k >= N ? 1 : 0, st = k - d * N;
            if (k > 0) {
              mbar_wait(&bb[B_H], ph_h); ph_h ^= 1;
              if constexpr (kTcHeads) {
                tc_fence_after();
                dense2_cell(k - 1);
              }
            }
            if (need_e1(k)) { mbar_wait(&bb[B_H1], ph_h1); ph_h1 ^= 1; }
            tc_fence_after();
            const uint32_t a0 = tmem + slot_col(agent_of(k));  // K blocks 0,1 from half 0 of the slot, 2,3 from half 1
            const unsigned char *wih_hi = sm_w + (d ? w.off_wih[1][0] : w.off_wih[0][0]);
            const unsigned char *wih_lo = sm_w + (d ? w.off_wih[1][1] : w.off_wih[0][1]);
            mma3_ts(tmem, a0, a0 + 16, wih_hi, wih_lo, kGateN * 16, 2, id_g, false);
            mma3_ts(tmem, a0 + 32, a0 + 48, wih_hi + 4 * kGateN * 16, wih_lo + 4 * kGateN * 16, kGateN * 16, 2, id_g, true);
            if (st > 0) mma3_ss(tmem, sm_h, sm_h + 8192, kChunkA, sm_w + (d ? w.off_whh[1][0] : w.off_whh[0][0]),
                                sm_w + (d ? w.off_whh[1][1] : w.off_whh[0][1]), kGateN * 16, 2, id_g, true);
            mma_commit(&bb[B_G]);
            // the next cell's dense1 goes behind this gate GEMM; its slot held the agent kSlots cells back, whose
            // last reader (with one slot: this gate GEMM) was issued before this point (the tensor pipe executes in
            // order)
            if (k + 1 < 2 * N && need_e1(k + 1)) dense1_cell(k + 1);
          }
          mbar_wait(&bb[B_H], ph_h); ph_h ^= 1;
          if constexpr (kTcHeads) {
            tc_fence_after();
            dense2_cell(2 * N - 1);
            mma_commit(&bb[B_L]);
          }
        }
      }
    }
    __syncwarp();
  } else {
    // =============================== the eight epilogue warps ===============================
    const int half = tid >> 7, own = half, row = tid & 127;
    const uint32_t lane_base = (uint32_t)(row & ~31) << 16;
    const float *b1 = reinterpret_cast<const float *>(sm_w + w.off_b1);
    const float *b2 = reinterpret_cast<const float *>(sm_w + w.off_b2);
    const float *w2f = reinterpret_cast<const float *>(sm_w + w.off_w2f);
    unsigned char *own_x = tile_smem(own), *own_h = own_x + xb;
    uint8_t *own_act = own_h + 16384;
    float *stage_obs = reinterpret_cast<float *>(own_x), *stage_rew = stage_obs + kRows * R;
    uint32_t ph_d1[2] = {0, 0}, ph_g[2] = {0, 0}, ph_l = 0;
    bool tma_pending = false;  // row 0: a bulk store of the staging buffer (= the obs operand buffer) may still be reading it
    // large teams: this CTA's dense2-share scratch, [tile][half][cell][pair of head entries][row]
    f2 *scr = (kJit || kXs) ? reinterpret_cast<f2 *>(w.scratch) + (size_t)blockIdx.x * tc2_scratch_f2_per_cta(N, APAD) : nullptr;
    bool have_w = false;  // the weight image (TMA bulk load issued at kernel start) is awaited behind the first operand phase
#ifdef MPE_TC_PHASES
    if (dbg && tid == 0 && blockIdx.x < 148) g_tc_timeline[blockIdx.x * 128 + 67] = clock64();
#endif
    for (int64_t pair = blockIdx.x; pair < npairs; pair += gridDim.x) {
#ifdef MPE_TC_PHASES
      if (dbg && tid == 0 && blockIdx.x < 148 && pair != blockIdx.x) g_tc_timeline[blockIdx.x * 128 + 68] = clock64();
#endif
      const int64_t tile = pair * 2 + own;                 // the tile this warpgroup owns (may not exist)
      const int64_t env0 = tile * kRows;
      const int64_t nb = FUSED ? s.B : io.B;
      const int valid = tile < ntiles ? (int)((nb - env0) < kRows ? (nb - env0) : kRows) : 0;
      const bool mine = row < valid;
      const int64_t b = env0 + row;
      [[maybe_unused]] const bool first_tile = pair == blockIdx.x && row == 0;
      for (int it = 0; it < T; ++it) {
        TL(half, 0);
        // ---- own tile: observations -> fp16 hi/lo A operands (large teams: the service warp streams them) ----
        if constexpr (!kJit) {
          Env<float, SC, N> e;
          float comm[2][10];
          if (FUSED && mine) {
            e.load(s, b);
            if (SC == kReference) {
#pragma unroll
              for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int k = 0; k < 10; ++k) comm[i][k] = s.comm[((int64_t)i * 10 + k) * s.B + b];
            }
          }
          if (FUSED) {
            // The previous step's TMA store drains the staging buffer while the state loads above are in flight;
            // only now, before the operand stores reuse that memory, does its issuer wait for the read to finish.
            if (tma_pending) bulk_wait_read_all();
            tma_pending = false;
            bar_sync_n(2 + own, 128);
          }
#pragma unroll
          for (int t = 0; t < N; ++t) {
            float xr[32];
#pragma unroll
            for (int k = 0; k < 32; ++k) xr[k] = 0.0f;
            if (FUSED) {
              if (mine) e.obs_row(t, xr, SC == kReference ? comm[1 - (t & 1)] : nullptr);
            } else if (mine) {
              const float *src = io.obs + b * R + t * D;
#pragma unroll
              for (int k = 0; k < 32; ++k)
                if (k < D) xr[k] = src[k];
            }
            unsigned char *xh = own_x + (size_t)(t * 2) * (Kx / 8) * kChunkA, *xl = xh + (size_t)(Kx / 8) * kChunkA;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              if (c * 8 < Kx) {
                const float v[8] = {xr[c * 8], xr[c * 8 + 1], xr[c * 8 + 2], xr[c * 8 + 3],
                                    xr[c * 8 + 4], xr[c * 8 + 5], xr[c * 8 + 6], xr[c * 8 + 7]};
                store_chunk_split(xh + c * kChunkA, xl + c * kChunkA, row, v);
              }
            }
          }
        }
        if constexpr (!kJit) {
          fence_proxy_async_smem();
          if constexpr (kTcHeads) tc_fence_before();  // the previous step's logit loads precede the next MMAs
          mbar_arrive(&bars[1 + own * B_PER_WG + B_X]);
        }

        if (!have_w) { mbar_wait(&bars[0], 0); have_w = true; }
        // FFMA heads: dense2 sums of the OWN tile's rows over this thread's 16 units, packed pairs of head entries
        // (large teams: just the bias, the shares come from the scratch rows).  Two-head actors add the bias after the
        // two warpgroups' sums: (own + other) + bias rounds the same whichever warpgroup owns the tile, so an env's
        // logits do not depend on the parity of its tile, i.e. on where it sits in the batch (HostRollout shards start
        // anywhere).  Unused with the heads on the tensor pipe, whose sums are the same MMAs for every tile.
        constexpr int NLG = kXs ? N : 1;
        f2 lgp[NLG][APAD / 2];
#pragma unroll
        for (int t = 0; t < NLG; ++t)
#pragma unroll
          for (int a = 0; a < APAD / 2; ++a) lgp[t][a] = kJit ? pk(b2[2 * a], b2[2 * a + 1]) : 0ull;

        // cell state of this thread's 16 units (2 chunks x 4 packed pairs), one set per tile
        f2 cA[2][4], cB[2][4];
#ifdef MPE_TC_PHASES  // per-phase cycle accounting of the pipeline (tools/tc_timeline.py); costs ~12 registers
        uint32_t acc[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0}, tlast = clock();
#define TS(i)                                   \
  do {                                          \
    if (dbg) {                                  \
      const uint32_t now = clock();             \
      acc[i] += now - tlast;                    \
      tlast = now;                              \
    }                                           \
  } while (0)
#else
#define TS(i)
#endif
        // E1(X): dense1 epilogue of this thread's 32 hidden columns of tile X's next cell
        auto E1 = [&](auto XT, int k) {
          constexpr int X = decltype(XT)::value;
          uint64_t *bb = bars + 1 + X * B_PER_WG;
          const uint32_t tmem = tmem_base + X * 256 + slot_col(agent_of(k)) + half * 32;
          TS(9);
          mbar_wait(&bb[B_D1], ph_d1[X]); ph_d1[X] ^= 1;
          tc_fence_after();
          TS(0);
          uint32_t v0[32];
          tmem_ld32(tmem + lane_base, v0);
          tmem_wait_ld();
          TS(1);
          dense1_half(v0, b1 + half * 32, tmem + lane_base, 16);  // in place: hi pairs, then lo pairs
          TS(2);
          tmem_wait_st();
          tc_fence_before();
          mbar_arrive(&bb[B_H1]);
          TS(3);
        };
        // C(X, k): LSTM cell k of tile X on this thread's 16 units; relu(h) to the tile's dense2 operand in TMEM, or
        // (FFMA heads) the dense2 share to lgp (own tile) or the scratch rows
        auto CC = [&](auto XT, int k, f2 (&c)[2][4]) {
          constexpr int X = decltype(XT)::value;
          const int d = k >= N ? 1 : 0, st = k - d * N;
          [[maybe_unused]] const int t = d == 0 ? st : N - 1 - st;
          uint64_t *bb = bars + 1 + X * B_PER_WG;
          const uint32_t tmem = tmem_base + X * 256;
          unsigned char *sm_h = tile_smem(X) + xb;
          if (st == 0) {
#pragma unroll
            for (int q = 0; q < 4; ++q) c[0][q] = c[1][q] = 0ull;
          }
          const float *bg = reinterpret_cast<const float *>(sm_w + w.off_bg) + d * kGateN + half * 64;
          [[maybe_unused]] const float *w2d = w2f + (d * kH + half * 16) * 16;
          [[maybe_unused]] f2 pl[APAD / 2];
          if constexpr (!kTcHeads) {
#pragma unroll
            for (int a = 0; a < APAD / 2; ++a) pl[a] = 0ull;
          }
          TS(9);
          mbar_wait(&bb[B_G], ph_g[X]); ph_g[X] ^= 1;
          tc_fence_after();
          TS(4);
          {
            // dense3 head requested (actor_forward with next_state): relu(h) of this thread's 16 units goes to
            // hcat[env][agent][dir * 32 + unit]; rows beyond the batch are skipped
            float *hc = nullptr;
            if constexpr (!FUSED) {
              if (io.hcat != nullptr) {
                const int64_t bx = (pair * 2 + X) * (int64_t)kRows + row;
                if (bx < io.B) hc = io.hcat + (bx * N + (d == 0 ? st : N - 1 - st)) * kHid + d * kH + half * 16;
              }
            }
            uint32_t va[32], vb[32];
            tmem_ld32(tmem + lane_base + half * 64, va);
            tmem_wait_ld();
            TS(5);
            tmem_ld32(tmem + lane_base + half * 64 + 32, vb);  // in flight during the first chunk's math
            if constexpr (kTcHeads) {
              // this thread's 16 units are K rows 16 half .. 16 half + 15 of the operand: hi columns 8 half .. 8 half + 7
              const uint32_t trelu = tmem + lane_base + kReluCol + half * 8;
              lstm_chunk_tc(va, bg, c[0], trelu, sm_h + (2 * half) * kChunkA, row, st < N - 1, hc);
              TS(6);
              tmem_wait_ld();
              TS(7);
              lstm_chunk_tc(vb, bg + 32, c[1], trelu + 4, sm_h + (2 * half + 1) * kChunkA, row, st < N - 1,
                            hc != nullptr ? hc + 8 : nullptr);
              tmem_wait_st();
            } else {
              lstm_chunk<APAD>(va, bg, w2d, c[0], pl, sm_h + (2 * half) * kChunkA, row, st < N - 1, hc);
              TS(6);
              tmem_wait_ld();
              TS(7);
              lstm_chunk<APAD>(vb, bg + 32, w2d + 8 * 16, c[1], pl, sm_h + (2 * half + 1) * kChunkA, row, st < N - 1,
                               hc != nullptr ? hc + 8 : nullptr);
            }
          }
          fence_proxy_async_smem();
          tc_fence_before();
          mbar_arrive(&bb[B_H]);
          TS(8);
          if constexpr (kJit) {
            // every cell's share goes to its own scratch row (no read-modify-write); the owner warpgroup completes
            // the logits from the four shares of an agent after the pipeline
            f2 *dst = scr + ((size_t)((X * 2 + half) * 2 * N + k) * (APAD / 2)) * kRows + row;
#pragma unroll
            for (int a = 0; a < APAD / 2; ++a) dst[a * kRows] = pl[a];
          } else if constexpr (kXs) {
            if (X == own) {
#pragma unroll
              for (int tt = 0; tt < NLG; ++tt)
                if (tt == t) {
#pragma unroll
                  for (int a = 0; a < APAD / 2; ++a) lgp[tt][a] = add2(lgp[tt][a], pl[a]);
                }
            } else {  // the other tile's rows: one scratch row per cell, summed by the owner
              f2 *dst = scr + ((size_t)((X * 2 + half) * 2 * N + k) * (APAD / 2)) * kRows + row;
#pragma unroll
              for (int a = 0; a < APAD / 2; ++a) dst[a * kRows] = pl[a];
            }
          }
        };
        // ---- the interleaved cell pipeline:  E1(A,0) | E1(B,k) C(A,k) E1(A,k+1) C(B,k) | ...  (tile A = 0, B = 1) ----
        using I0 = std::integral_constant<int, 0>;
        using I1 = std::integral_constant<int, 1>;
        TL(half, 1);
        E1(I0{}, 0);
#pragma unroll 1
        for (int k = 0; k < 2 * N; ++k) {
          TL(half, 2 + 2 * k);
          if (need_e1(k)) E1(I1{}, k);
          CC(I0{}, k, cA);
          TL(half, 3 + 2 * k);
          if (k + 1 < 2 * N && need_e1(k + 1)) E1(I0{}, k + 1);
          CC(I1{}, k, cB);
        }
        TL(half, 28);
#ifdef MPE_TC_PHASES
        if (dbg && first_tile) {
#pragma unroll
          for (int i = 0; i < 10; ++i) g_tc_timeline[blockIdx.x * 128 + 96 + half * 10 + i] = acc[i];
        }
#endif
        if constexpr (kTcHeads) {
          mbar_wait(&bars[1 + own * B_PER_WG + B_L], ph_l); ph_l ^= 1;
          tc_fence_after();
        } else {
          bar_sync_n(1, 256);  // the scratch shares of both warpgroups are complete
        }
        TL(half, 14);

        // ---- own tile: Gumbel-max sampling ----
        int au[N], ac[N];
        if constexpr (kJit) {
          // groups of G agents: logits = bias + the four scratch shares (two warpgroups x two directions); the G * 2
          // Philox blocks and the G * 5 Gumbel transforms of a group run in lock-step
          constexpr int G = (N % 3 == 0) ? 3 : 2, NQ = APAD / 4;
#pragma unroll 1
          for (int t0 = 0; t0 < N; t0 += G) {
            float lgt[G][APAD], gn[G][APAD];
#pragma unroll
            for (int u = 0; u < G; ++u) {
              const int t = t0 + u, kf = t, kb = 2 * N - 1 - t;
              auto at = [&](int hf, int k) { return scr + ((size_t)((own * 2 + hf) * 2 * N + k) * (APAD / 2)) * kRows + row; };
#pragma unroll
              for (int a = 0; a < APAD / 2; ++a) {
                const f2 sf = add2(at(0, kf)[a * kRows], at(1, kf)[a * kRows]);
                const f2 sb = add2(at(0, kb)[a * kRows], at(1, kb)[a * kRows]);
                upk(add2(add2(lgp[0][a], sf), sb), lgt[u][2 * a], lgt[u][2 * a + 1]);
              }
#pragma unroll
              for (int a = 0; a < APAD; ++a) gn[u][a] = 0.0f;
            }
            if (io.gumbel != nullptr) {
              if (mine) {
#pragma unroll
                for (int u = 0; u < G; ++u)
#pragma unroll
                  for (int a = 0; a < APAD; ++a)
                    if (a < w.A) gn[u][a] = io.gumbel[(b * N + t0 + u) * w.A + a];
              }
            } else {
              uint4 c[G * NQ];
#pragma unroll
              for (int u = 0; u < G; ++u)
#pragma unroll
                for (int jj = 0; jj < NQ; ++jj)
                  c[u * NQ + jj] = philox_counter((uint64_t)(io.gid0 + b), (uint32_t)io.step, kDomainGumbel, (t0 + u) * 8 + jj);
              philox4x32_10_batch<G * NQ>(c, philox_key(io.seed));
              if (w.A == 5) {
                uint32_t r[G * 5];
                float g[G * 5];
#pragma unroll
                for (int u = 0; u < G; ++u) {
                  r[u * 5 + 0] = c[u * NQ].x; r[u * 5 + 1] = c[u * NQ].y; r[u * 5 + 2] = c[u * NQ].z;
                  r[u * 5 + 3] = c[u * NQ].w; r[u * 5 + 4] = c[u * NQ + 1].x;
                }
                bits_to_gumbel_batch<G * 5>(r, g);
#pragma unroll
                for (int u = 0; u < G; ++u)
#pragma unroll
                  for (int a = 0; a < 5; ++a) gn[u][a] = g[u * 5 + a];
              } else {
#pragma unroll
                for (int u = 0; u < G; ++u) {
                  uint32_t r[APAD];
                  float g[APAD];
#pragma unroll
                  for (int jj = 0; jj < NQ; ++jj) {
                    r[4 * jj] = c[u * NQ + jj].x; r[4 * jj + 1] = c[u * NQ + jj].y;
                    r[4 * jj + 2] = c[u * NQ + jj].z; r[4 * jj + 3] = c[u * NQ + jj].w;
                  }
                  bits_to_gumbel_batch<APAD>(r, g);
#pragma unroll
                  for (int a = 0; a < APAD; ++a) gn[u][a] = a < w.A ? g[a] : 0.0f;
                }
              }
            }
#pragma unroll
            for (int u = 0; u < G; ++u) {
              const int t = t0 + u;
              int bu = 0, bc = 0;
              float best = lgt[u][0] + gn[u][0];
#pragma unroll
              for (int a = 1; a < APAD; ++a) {
                const float z = lgt[u][a] + gn[u][a];
                if (a < w.A0 && z > best) { best = z; bu = a; }
              }
              if (w.A1 > 0) {
                float bcv = -INFINITY;
#pragma unroll
                for (int a = 0; a < APAD; ++a) {
                  const float z = lgt[u][a] + gn[u][a];
                  if (a >= w.A0 && a < w.A && z > bcv) { bcv = z; bc = a - w.A0; }
                }
              }
              own_act[(row * N + t) * 2] = (uint8_t)bu;
              own_act[(row * N + t) * 2 + 1] = (uint8_t)bc;
              if (mine && io.logits != nullptr) {
#pragma unroll
                for (int a = 0; a < APAD; ++a)
                  if (a < w.A) io.logits[(b * N + t) * w.A + a] = lgt[u][a];
              }
            }
          }
        } else {
          const uint64_t step = FUSED ? ro.step0 + (uint64_t)it : io.step;
          const uint64_t seed = FUSED ? s.seed : io.seed;
          const int64_t gid0 = FUSED ? s.gid0 : io.gid0;
          // heads on the tensor pipe: the 16-fold logit sums of agent t in columns 8t..8t+7, loaded behind the noise
          [[maybe_unused]] uint32_t lv[N][8];
          if constexpr (kTcHeads) {
#pragma unroll
            for (int t = 0; t < N; ++t) tmem_ld8(tmem_base + own * 256 + lane_base + kLogitCol + 8 * t, lv[t]);
          }
          // Gumbel noise of all N agents of this row up front: the N * APAD/4 Philox blocks advance together and
          // the log chains of the values run in lock-step (see bits_to_gumbel_batch)
          float gn[N][APAD];
#pragma unroll
          for (int t = 0; t < N; ++t)
#pragma unroll
            for (int a = 0; a < APAD; ++a) gn[t][a] = 0.0f;
          if (!FUSED && io.gumbel != nullptr) {
            if (mine) {
#pragma unroll
              for (int t = 0; t < N; ++t)
#pragma unroll
                for (int a = 0; a < APAD; ++a)
                  if (a < w.A) gn[t][a] = io.gumbel[(b * N + t) * w.A + a];
            }
          } else {
            constexpr int NQ = APAD / 4;
            uint4 c[N * NQ];
#pragma unroll
            for (int t = 0; t < N; ++t)
#pragma unroll
              for (int jj = 0; jj < NQ; ++jj)
                c[t * NQ + jj] = philox_counter((uint64_t)(gid0 + b), (uint32_t)step, kDomainGumbel, t * 8 + jj);
            philox4x32_10_batch<N * NQ>(c, philox_key(seed));
            if (w.A == 5) {  // the movement head of every supported scenario: exactly the 5 used values per agent
              uint32_t r[N * 5];
              float g[N * 5];
#pragma unroll
              for (int t = 0; t < N; ++t) {
                r[t * 5 + 0] = c[t * NQ].x; r[t * 5 + 1] = c[t * NQ].y; r[t * 5 + 2] = c[t * NQ].z;
                r[t * 5 + 3] = c[t * NQ].w; r[t * 5 + 4] = c[t * NQ + 1].x;
              }
              bits_to_gumbel_batch<N * 5>(r, g);
#pragma unroll
              for (int t = 0; t < N; ++t)
#pragma unroll
                for (int a = 0; a < 5; ++a) gn[t][a] = g[t * 5 + a];
            } else {
#pragma unroll
              for (int t = 0; t < N; ++t) {
                uint32_t r[APAD];
                float g[APAD];
#pragma unroll
                for (int jj = 0; jj < NQ; ++jj) {
                  r[4 * jj] = c[t * NQ + jj].x; r[4 * jj + 1] = c[t * NQ + jj].y;
                  r[4 * jj + 2] = c[t * NQ + jj].z; r[4 * jj + 3] = c[t * NQ + jj].w;
                }
                bits_to_gumbel_batch<APAD>(r, g);
#pragma unroll
                for (int a = 0; a < APAD; ++a) gn[t][a] = a < w.A ? g[a] : 0.0f;
              }
            }
          }
          if constexpr (kTcHeads) tmem_wait_ld();
#pragma unroll
          for (int t = 0; t < N; ++t) {
            float z[APAD];
            float lgt[APAD];
            if constexpr (kTcHeads) {
#pragma unroll
              for (int a = 0; a < APAD; ++a) lgt[a] = fmaf(__uint_as_float(lv[t][a]), kWInv, b2[a]);  // x 1/16: exact
            } else {
#pragma unroll
              for (int a = 0; a < APAD / 2; ++a) {
                const f2 *sf = scr + ((size_t)((own * 2 + (1 - half)) * 2 * N + t) * (APAD / 2) + a) * kRows + row;
                const f2 *sb = scr + ((size_t)((own * 2 + (1 - half)) * 2 * N + (2 * N - 1 - t)) * (APAD / 2) + a) * kRows + row;
                upk(add2(add2(lgp[t][a], add2(*sf, *sb)), pk(b2[2 * a], b2[2 * a + 1])), lgt[2 * a], lgt[2 * a + 1]);
              }
            }
            const int64_t orow = b * N + t;
#pragma unroll
            for (int a = 0; a < APAD; ++a) z[a] = a < w.A ? lgt[a] + gn[t][a] : 0.0f;
            int bu = 0, bc = 0;
            float best = z[0];
#pragma unroll
            for (int a = 1; a < APAD; ++a)
              if (a < w.A0 && z[a] > best) { best = z[a]; bu = a; }
            if (w.A1 > 0) {
              float bcv = -INFINITY;
#pragma unroll
              for (int a = 0; a < APAD; ++a)
                if (a >= w.A0 && a < w.A && z[a] > bcv) { bcv = z[a]; bc = a - w.A0; }
            }
            au[t] = bu; ac[t] = bc;
            TL(half, 15 + t);
            own_act[(row * N + t) * 2] = (uint8_t)bu;
            own_act[(row * N + t) * 2 + 1] = (uint8_t)bc;
            if (!FUSED && mine && io.logits != nullptr) {
#pragma unroll
              for (int a = 0; a < APAD; ++a)
                if (a < w.A) io.logits[orow * w.A + a] = lgt[a];
            }
          }
        }

        TL(half, 29);
        if constexpr (FUSED) {
          // ---- own tile: World.step + reward + outputs for env row `row` ----
          const int64_t toff = (int64_t)it * s.B;
          bool do_reset = false;
          Env<float, SC, N> e;
          float comm[2][10];
          double ret = 0.0, n_ep = 0.0, n_steps = 0.0;
          if (mine) {
            e.load(s, b);
            TL(half, 18);
            e.physics(au, s);
            TL(half, 19);
            if (SC == kReference) {
#pragma unroll
              for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int k = 0; k < 10; ++k) comm[i][k] = k == ac[i] ? 1.0f : 0.0f;
            }
            float r[N];
            int coll[N], occ;
            float md;
            e.reward(r, coll, occ, md, s);
            if constexpr (INFO) {  // the values and layout of mpe_step's info_i / info_f, at [it][b]
              if (ro.info_i != nullptr) {
                int32_t *ii = ro.info_i + (toff + b) * (N + 1);
#pragma unroll
                for (int i = 0; i < N; ++i) ii[i] = coll[i];
                ii[N] = occ;
              }
              if (ro.info_f != nullptr) ro.info_f[toff + b] = md;
            }
            float sum = 0.0f;
#pragma unroll
            for (int i = 0; i < N; ++i) { sum += r[i]; stage_rew[row * N + i] = r[i]; }
            const float ep_ret = s.ep_ret[b] + sum;
            const int ts = s.tstep[b] + 1;
            do_reset = max_episode_len > 0 && ts >= max_episode_len;
#pragma unroll
            for (int i = 0; i < N; ++i) e.obs_row(i, stage_obs + row * R + i * D, SC == kReference ? comm[1 - (i & 1)] : nullptr);
            if (do_reset) {
              ret = (double)ep_ret; n_ep = 1.0; n_steps = (double)ts;
              s.ep_ret[b] = 0.0f; s.tstep[b] = 0;
            } else {
              s.ep_ret[b] = ep_ret; s.tstep[b] = ts;
            }
          }
          TL(half, 21);
          fold_stats(s.stats, ret, n_ep, n_steps);
          float *g_obs = (ro.obs_next != nullptr && valid > 0) ? ro.obs_next + (toff + env0) * R : nullptr;
          float *g_rew = (ro.rew != nullptr && valid > 0) ? ro.rew + (toff + env0) * N : nullptr;
          const bool tma_ok = valid == kRows && ((reinterpret_cast<uintptr_t>(g_obs) | reinterpret_cast<uintptr_t>(g_rew)) & 15) == 0;
          if (tma_ok) fence_proxy_async_smem();
          bar_sync_n(2 + own, 128);
          TL(half, 22);
          if (g_obs != nullptr || g_rew != nullptr) {
            if (tma_ok) {
              if (row == 0) {
                if (g_obs != nullptr) bulk_store(g_obs, stage_obs, kRows * R * 4);
                if (g_rew != nullptr) bulk_store(g_rew, stage_rew, kRows * N * 4);
                bulk_commit();
              }
            } else {
              if (g_obs != nullptr)
                for (int i = row; i < valid * R; i += 128) g_obs[i] = stage_obs[i];
              if (g_rew != nullptr)
                for (int i = row; i < valid * N; i += 128) g_rew[i] = stage_rew[i];
            }
          }
          if (ro.act_u != nullptr)
            for (int i = row; i < valid * N; i += 128) ro.act_u[(toff + env0) * N + i] = own_act[i * 2];
          if (ro.act_c != nullptr)
            for (int i = row; i < valid * N; i += 128) ro.act_c[(toff + env0) * N + i] = own_act[i * 2 + 1];
          if (mine) {
            if (do_reset) {  // experiments/run.py:59-60
              const uint32_t ep = s.episode[b] + 1u;
              s.episode[b] = ep;
              e.reset(s.seed, (uint64_t)(s.gid0 + b), ep);
              e.store_world(s, b);
              if (SC == kReference) {
#pragma unroll
                for (int i = 0; i < 2; ++i)
#pragma unroll
                  for (int k = 0; k < 10; ++k) comm[i][k] = 0.0f;
              }
            }
            e.store_agents(s, b);
            if (SC == kReference) {
#pragma unroll
              for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int k = 0; k < 10; ++k) s.comm[((int64_t)i * 10 + k) * s.B + b] = comm[i][k];
            }
          }
          TL(half, 23);
          if (row == 0 && tma_ok && (g_obs != nullptr || g_rew != nullptr)) tma_pending = true;
        } else {
          bar_sync_n(2 + own, 128);
          const int rows = valid * N;
          if (io.act_u != nullptr)
            for (int i = row; i < rows; i += 128) io.act_u[env0 * N + i] = own_act[i * 2];
          if (io.act_c != nullptr)
            for (int i = row; i < rows; i += 128) io.act_c[env0 * N + i] = own_act[i * 2 + 1];
          if (io.onehot != nullptr)
            for (int i = row; i < rows * w.A; i += 128) {
              const int rr = i / w.A, a = i - rr * w.A;
              const bool hot = a < w.A0 ? (a == own_act[rr * 2]) : (a - w.A0 == own_act[rr * 2 + 1]);
              io.onehot[env0 * N * w.A + i] = hot ? 1.0f : 0.0f;
            }
        }
        TL(half, 30);
        bar_sync_n(1, 256);  // action buffers of both tiles are free again (staging: see tma_pending)
        TL(half, 31);
      }
    }
    if (tma_pending) bulk_wait_read_all();  // shared memory must stay valid until the last bulk store has read it
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 8) tmem_free(tmem_base, 512);
#ifdef MPE_TC_PHASES
  if (dbg && threadIdx.x == 0 && blockIdx.x < 148) {
    unsigned long long gt;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
    g_tc_timeline[blockIdx.x * 128 + 65] = gt;
    g_tc_timeline[blockIdx.x * 128 + 69] = clock64();
  }
#endif
}

// ------------------------------------------------------------------------------------------------
// launch
// ------------------------------------------------------------------------------------------------
static int tc_debug_flag() {
  static const int dbg = getenv("MPE_TC_TIMELINE") != nullptr ? 1 : 0;
  return dbg;
}

// Per-launch host work is kept to the launch itself (the fused step is a ~60 us kernel): one cudaGetDevice, everything
// derived from the device is cached (launch.h).
template <int SC, int N, bool FUSED, int APAD, bool INFO = false>
static cudaError_t launch_tc2_t(const EnvState<float> &s, const TcDev &w, const ActorIO &io, const RolloutIO &ro,
                                int max_episode_len, int64_t nenvs, cudaStream_t st) {
  const int dev = current_device();
  const size_t smem = tc2_smem_bytes(w.bytes, N, w.Kx);
  if (smem > 227 * 1024) return cudaErrorInvalidValue;  // tc_*_supported rule these out
  cudaError_t e = ensure_smem<k_tc2<SC, N, FUSED, APAD, INFO>>(smem, dev);
  if (e != cudaSuccess) return e;
  const int64_t ntiles = (nenvs + kRows - 1) / kRows;
  const int nsm = sm_count(dev);
  const int64_t pairs = (ntiles + 1) / 2;
  const int grid = (int)(pairs < nsm ? pairs : nsm);
  k_tc2<SC, N, FUSED, APAD, INFO><<<grid, tc2_threads(N), smem, st>>>(s, w, io, ro, max_episode_len, ntiles, tc_debug_flag());
  return cudaGetLastError();
}

bool tc_actor_supported(const TcDev &w, int N) {
  // teams of > 3 agents keep one head of <= 8 entries (launch_actor_forward_tc); wider heads go to the FFMA kernel
  return tc_supported(w) && (N == 2 || N == 3 || ((N == 4 || N == 6 || N == 8 || N == 9 || N == 12) && w.A <= 8 && w.scratch != nullptr));
}
bool tc_rollout_supported(const TcDev &w, int N) {
  // one kernel for all T steps: every agent of an env in one thread's registers
  return tc_supported(w) && (N == 2 || N == 3);
}
size_t tc_scratch_floats(int sm_count) {
  // the larger of k_tc2's per-cell shares for the instantiated large teams (N <= 12, one head of <= 8 entries) and
  // for the two-head small teams (N <= 3, 16 entries)
  const size_t v2 = (size_t)sm_count * tc2_scratch_f2_per_cta(12, 8) * 2, v3 = (size_t)sm_count * tc2_scratch_f2_per_cta(3, 16) * 2;
  return v2 > v3 ? v2 : v3;
}

cudaError_t launch_actor_forward_tc(const TcDev &w, const ActorIO &io, cudaStream_t st) {
  EnvState<float> s{};
  RolloutIO ro;
  const bool wide = w.A > 8;
  switch (io.N) {
    case 2: return wide ? launch_tc2_t<kSpread, 2, false, 16>(s, w, io, ro, 0, io.B, st)
                        : launch_tc2_t<kSpread, 2, false, 8>(s, w, io, ro, 0, io.B, st);
    case 3: return wide ? launch_tc2_t<kSpread, 3, false, 16>(s, w, io, ro, 0, io.B, st)
                        : launch_tc2_t<kSpread, 3, false, 8>(s, w, io, ro, 0, io.B, st);
    case 4: return wide ? cudaErrorInvalidValue : launch_tc2_t<kSpread, 4, false, 8>(s, w, io, ro, 0, io.B, st);
    case 6: return wide ? cudaErrorInvalidValue : launch_tc2_t<kSpread, 6, false, 8>(s, w, io, ro, 0, io.B, st);
    case 8: return wide ? cudaErrorInvalidValue : launch_tc2_t<kSpread, 8, false, 8>(s, w, io, ro, 0, io.B, st);
    case 9: return wide ? cudaErrorInvalidValue : launch_tc2_t<kSpread, 9, false, 8>(s, w, io, ro, 0, io.B, st);
    case 12: return wide ? cudaErrorInvalidValue : launch_tc2_t<kSpread, 12, false, 8>(s, w, io, ro, 0, io.B, st);
    default: return cudaErrorInvalidValue;
  }
}

template <int SC, int N, int APAD>
static cudaError_t launch_rollout_tc_t(const EnvState<float> &s, const TcDev &w, const RolloutIO &ro, int max_episode_len,
                                       cudaStream_t st) {
  ActorIO io;
  if (ro.info_i != nullptr || ro.info_f != nullptr)
    return launch_tc2_t<SC, N, true, APAD, true>(s, w, io, ro, max_episode_len, s.B, st);
  return launch_tc2_t<SC, N, true, APAD>(s, w, io, ro, max_episode_len, s.B, st);
}

cudaError_t launch_rollout_tc(const EnvStateAny &a, const TcDev &w, const RolloutIO &ro, cudaStream_t st) {
  EnvState<float> s = typed<float>(a);
  s.track = 1;  // the fused rollout always keeps the episode counters (mpe_track_returns)
  const int L = a.max_episode_len;
  if (a.scenario == kReference) return launch_rollout_tc_t<kReference, 2, 16>(s, w, ro, L, st);
  if (a.scenario == kSpeaker) return launch_rollout_tc_t<kSpeaker, 2, 8>(s, w, ro, L, st);
  if (a.N == 2) return launch_rollout_tc_t<kSpread, 2, 8>(s, w, ro, L, st);
  if (a.N == 3) return launch_rollout_tc_t<kSpread, 3, 8>(s, w, ro, L, st);
  return cudaErrorInvalidValue;
}

}  // namespace mpe

// debug-only export (not part of include/mpe_b200.h)
extern "C" __attribute__((visibility("default"))) int mpe_debug_tc_timeline(unsigned long long *out, int n) {
  return (int)cudaMemcpyFromSymbol(out, mpe::g_tc_timeline, sizeof(unsigned long long) * (size_t)n);
}
