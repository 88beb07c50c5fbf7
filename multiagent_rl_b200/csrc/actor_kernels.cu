// Actor forward (dense1 -> BiLSTM over the agent axis -> dense2 heads -> hard Gumbel sample), fp32 SIMT, and the
// dense3 head that follows the tensor-core forward.
//
// Reference rows: rls/model/ac_network_multi_gumbel.py:52-67 (forward), :7-21 (TimeDistributed),
// rls/model/ac_network_model_multi_gumbel.py:49,65 (dense3 head),
// rls/agent/multiagent/ddpg_gumbel_fix.py:86-116 (get_exploration_action, gumbel_softmax hard=True).
//
// Shape of the computation: per env the LSTM is N sequential steps of a [96 -> 128] GEMV per
// direction; batching TB envs turns each step into a [TB x 96] x [96 x 128] GEMM whose B operand
// (the weights, 104 KB fp32) is identical for every env.  So: one persistent CTA per SM keeps the
// whole packed weight blob resident in shared memory (loaded once with a TMA bulk copy) and walks
// over tiles of TB envs.  Activations live in shared memory k-major ([k][env]) so that a thread's RT
// rows are one or two 16 B loads and a warp's A reads are broadcasts.  256 threads = 2 directions x
// 16 unit-groups x 8 row-groups; a thread owns RT rows x (4 gates x 2 units) = RT x 8 accumulators and
// the cell state of those (row, unit) pairs for the whole sequence, so c never leaves registers.
#include <cmath>

#include "actor_cell.cuh"
#include "actor_launch.h"
#include "common.cuh"
#include "launch.h"

namespace mpe {

constexpr int kActorThreads = 256;

// ------------------------------------------------------------------------------------------------
// host: blob layout (packed by pack_kernels.cu)
// ------------------------------------------------------------------------------------------------
static int round_up(int x, int m) { return (x + m - 1) / m * m; }

void actor_layout(int D, int A0, int A1, bool has_model, ActorDev *o) {
  o->D = D; o->A0 = A0; o->A1 = A1; o->A = A0 + A1;
  o->Apad = round_up(o->A, 4);
  o->Dpad = round_up(D, 4);
  o->has_model = has_model ? 1 : 0;
  int off = 0;
  o->off_wg[0] = off; off += kGateK * kGateN;
  o->off_wg[1] = off; off += kGateK * kGateN;
  o->off_bg = off; off += 2 * kGateN;
  o->off_w1 = off; off += round_up(D * kHid, 4);
  o->off_b1 = off; off += kHid;
  o->off_w2 = off; off += kHid * o->Apad;
  o->off_b2 = off; off += o->Apad;
  o->smem_floats = (size_t)round_up(off, 32);  // the dense3 head stays in global memory (L2): not on the acting path
  off = (int)o->smem_floats;
  o->off_w3 = off; off += has_model ? kHid * o->Dpad : 0;
  o->off_b3 = off; off += has_model ? o->Dpad : 0;
  o->blob_floats = (size_t)round_up(off, 32);
}

// ------------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------------
// sigmoid_f / tanh_f: actor_cell.cuh

template <int RT>
__device__ __forceinline__ void load_rows(const float *p, float (&a)[RT]) {
  if constexpr (RT == 8) {
    const float4 u = *reinterpret_cast<const float4 *>(p), v = *reinterpret_cast<const float4 *>(p + 4);
    a[0] = u.x; a[1] = u.y; a[2] = u.z; a[3] = u.w; a[4] = v.x; a[5] = v.y; a[6] = v.z; a[7] = v.w;
  } else if constexpr (RT == 4) {
    const float4 u = *reinterpret_cast<const float4 *>(p);
    a[0] = u.x; a[1] = u.y; a[2] = u.z; a[3] = u.w;
  } else {
    const float2 u = *reinterpret_cast<const float2 *>(p);
    a[0] = u.x; a[1] = u.y;
  }
}
template <int RT>
__device__ __forceinline__ void store_rows(float *p, const float (&a)[RT]) {
  if constexpr (RT == 8) {
    *reinterpret_cast<float4 *>(p) = make_float4(a[0], a[1], a[2], a[3]);
    *reinterpret_cast<float4 *>(p + 4) = make_float4(a[4], a[5], a[6], a[7]);
  } else if constexpr (RT == 4) {
    *reinterpret_cast<float4 *>(p) = make_float4(a[0], a[1], a[2], a[3]);
  } else {
    *reinterpret_cast<float2 *>(p) = make_float2(a[0], a[1]);
  }
}

// acc[RT][8] += A[k][rows] * W[k][cols] over K contraction steps (A, W in shared memory, k-major)
template <int RT>
__device__ __forceinline__ void gate_gemm(const float *__restrict__ A, int lda, const float *__restrict__ W, int K,
                                          float (&acc)[RT][8]) {
#pragma unroll 4
  for (int k = 0; k < K; ++k) {
    float a[RT];
    load_rows<RT>(A + k * lda, a);
    const float4 w0 = *reinterpret_cast<const float4 *>(W + k * kGateN);
    const float4 w1 = *reinterpret_cast<const float4 *>(W + k * kGateN + 4);
    const float w[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
    for (int r = 0; r < RT; ++r)
#pragma unroll
      for (int c = 0; c < 8; ++c) acc[r][c] = fmaf(a[r], w[c], acc[r][c]);
  }
}

__device__ __forceinline__ void bar_named(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

template <int N, int TB, int PAD>
struct ActorSmem {
  static constexpr int TBP = TB + PAD;
  static constexpr int RT = TB / 8;
  float *w, *h1, *hc, *obs, *rew;  // rew: no reader; dropping it moves sm.act, a layout change to measure on its own
  int *act;
  uint64_t *bars;
  __host__ __device__ static size_t bytes(size_t blob_floats, int D) {
    size_t f = blob_floats + 2 * (size_t)N * kHid * TBP + (size_t)((TB * N * D + 31) / 32 * 32) + (size_t)TB * N;
    return f * sizeof(float) + (size_t)TB * N * 2 * sizeof(int) + 2 * sizeof(uint64_t) + 16;
  }
  __device__ void carve(float *base, size_t blob_floats, int D) {
    w = base;
    h1 = w + blob_floats;
    hc = h1 + (size_t)N * kHid * TBP;
    obs = hc + (size_t)N * kHid * TBP;
    rew = obs + (TB * N * D + 31) / 32 * 32;
    act = reinterpret_cast<int *>(rew + TB * N);
    bars = reinterpret_cast<uint64_t *>((reinterpret_cast<uintptr_t>(act + TB * N * 2) + 15) & ~(uintptr_t)15);
  }
};

// dense1 + BiLSTM + heads + sampling for one tile whose observations are in sm.obs ([TB][N*D]).
// On return sm.act[(e*N + t)*2 + {0,1}] holds the sampled indices; global outputs (if any) are written
// for the `valid` leading envs of the tile.
template <int N, int TB, int PAD>
__device__ __forceinline__ void actor_tile(const ActorDev &w, const ActorSmem<N, TB, PAD> &sm, const ActorIO &io,
                                           int64_t env0, int valid, uint64_t step) {
  constexpr int TBP = TB + PAD, RT = TB / 8;
  const int tid = threadIdx.x;
  const int D = w.D, ND = N * w.D;

  // ---- dense1: h1[t][j][e] = relu(b1[j] + sum_k obs[e][t][k] * W1[k][j]) ----
  {
    constexpr int G = kActorThreads / TB;  // j-groups
    constexpr int JG = kHid / G;           // outputs per thread (multiple of 4)
    const int e = tid % TB, j0 = (tid / TB) * JG;
    const float *W1 = sm.w + w.off_w1, *b1 = sm.w + w.off_b1;
#pragma unroll 1
    for (int t = 0; t < N; ++t) {
      float acc[JG];
#pragma unroll
      for (int j = 0; j < JG; ++j) acc[j] = b1[j0 + j];
      const float *x = sm.obs + e * ND + t * D;
#pragma unroll 2
      for (int k = 0; k < D; ++k) {
        const float xk = x[k];
#pragma unroll
        for (int j = 0; j < JG; j += 4) {
          const float4 wv = *reinterpret_cast<const float4 *>(W1 + k * kHid + j0 + j);
          acc[j] = fmaf(xk, wv.x, acc[j]); acc[j + 1] = fmaf(xk, wv.y, acc[j + 1]);
          acc[j + 2] = fmaf(xk, wv.z, acc[j + 2]); acc[j + 3] = fmaf(xk, wv.w, acc[j + 3]);
        }
      }
#pragma unroll
      for (int j = 0; j < JG; ++j) sm.h1[(t * kHid + j0 + j) * TBP + e] = fmaxf(acc[j], 0.0f);
    }
  }
  __syncthreads();

  // ---- BiLSTM over the agent axis ----
  {
    const int dir = tid >> 7, q = tid & 127, ug = q & 15, rg = q >> 4;
    const float *Wg = sm.w + w.off_wg[dir] + ug * 8;
    const float *bg = sm.w + w.off_bg + dir * kGateN + ug * 8;
    float c[RT][2];
#pragma unroll
    for (int r = 0; r < RT; ++r) c[r][0] = c[r][1] = 0.0f;
#pragma unroll 1
    for (int s = 0; s < N; ++s) {
      const int t = dir == 0 ? s : N - 1 - s;
      float acc[RT][8];
      {
        const float4 b0 = *reinterpret_cast<const float4 *>(bg), b1 = *reinterpret_cast<const float4 *>(bg + 4);
#pragma unroll
        for (int r = 0; r < RT; ++r) {
          acc[r][0] = b0.x; acc[r][1] = b0.y; acc[r][2] = b0.z; acc[r][3] = b0.w;
          acc[r][4] = b1.x; acc[r][5] = b1.y; acc[r][6] = b1.z; acc[r][7] = b1.w;
        }
      }
      gate_gemm<RT>(sm.h1 + (t * kHid) * TBP + rg * RT, TBP, Wg, kHid, acc);
      if (s > 0) {
        const int tp = dir == 0 ? t - 1 : t + 1;
        gate_gemm<RT>(sm.hc + (tp * kHid + dir * kH) * TBP + rg * RT, TBP, Wg + kHid * kGateN, kH, acc);
      }
      // packed columns: [i0 i1 f0 f1 g0 g1 o0 o1] for units (ug, ug+16)
#pragma unroll
      for (int uu = 0; uu < 2; ++uu) {
        float h[RT];
#pragma unroll
        for (int r = 0; r < RT; ++r) {
          const float ig = sigmoid_f(acc[r][0 + uu]), fg = sigmoid_f(acc[r][2 + uu]);
          const float gg = tanh_f(acc[r][4 + uu]), og = sigmoid_f(acc[r][6 + uu]);
          c[r][uu] = fmaf(fg, c[r][uu], ig * gg);
          h[r] = og * tanh_f(c[r][uu]);
        }
        store_rows<RT>(sm.hc + (t * kHid + dir * kH + ug + 16 * uu) * TBP + rg * RT, h);
      }
      bar_named(1 + dir, 128);  // the two directions never read each other's rows inside the loop
    }
  }
  __syncthreads();

  // ---- heads on relu(hcat), Gumbel-max sampling ----
  if (tid < TB * N) {
    const int e = tid % TB, t = tid / TB;
    const int A = w.A, Apad = w.Apad, A0 = w.A0;
    const float *W2 = sm.w + w.off_w2, *b2 = sm.w + w.off_b2;
    float lg[kActorMaxA];
#pragma unroll
    for (int a = 0; a < kActorMaxA; ++a) lg[a] = a < Apad ? b2[a] : 0.0f;
    const float *hrow = sm.hc + (t * kHid) * TBP + e;
#pragma unroll 4
    for (int k = 0; k < kHid; ++k) {
      const float hk = fmaxf(hrow[k * TBP], 0.0f);
#pragma unroll
      for (int a = 0; a < kActorMaxA; a += 4) {
        if (a < Apad) {
          const float4 wv = *reinterpret_cast<const float4 *>(W2 + k * Apad + a);
          lg[a] = fmaf(hk, wv.x, lg[a]); lg[a + 1] = fmaf(hk, wv.y, lg[a + 1]);
          lg[a + 2] = fmaf(hk, wv.z, lg[a + 2]); lg[a + 3] = fmaf(hk, wv.w, lg[a + 3]);
        }
      }
    }
    const bool ok = e < valid;
    const int64_t row = (env0 + e) * N + t;
    float z[kActorMaxA];
    if (io.gumbel != nullptr) {
#pragma unroll
      for (int a = 0; a < kActorMaxA; ++a) z[a] = (a < A && ok) ? lg[a] + io.gumbel[row * A + a] : lg[a];
    } else {
#pragma unroll
      for (int j = 0; j < kActorMaxA / 4; ++j) {
        if (4 * j < A) {
          const uint4 r = philox_raw(io.seed, (uint64_t)(io.gid0 + env0 + e), (uint32_t)step, kDomainGumbel, t * 8 + j);
          z[4 * j] = lg[4 * j] + bits_to_gumbel(r.x); z[4 * j + 1] = lg[4 * j + 1] + bits_to_gumbel(r.y);
          z[4 * j + 2] = lg[4 * j + 2] + bits_to_gumbel(r.z); z[4 * j + 3] = lg[4 * j + 3] + bits_to_gumbel(r.w);
        }
      }
    }
    int au = 0, ac = 0;
    float best = z[0];
#pragma unroll
    for (int a = 1; a < kActorMaxA; ++a)
      if (a < A0 && z[a] > best) { best = z[a]; au = a; }
    if (w.A1 > 0) {
      float bc = -INFINITY;
      ac = 0;
#pragma unroll
      for (int a = 0; a < kActorMaxA; ++a)
        if (a >= A0 && a < A && z[a] > bc) { bc = z[a]; ac = a - A0; }
    }
    sm.act[(e * N + t) * 2] = au;
    sm.act[(e * N + t) * 2 + 1] = ac;
    if (ok && io.logits != nullptr) {
#pragma unroll
      for (int a = 0; a < kActorMaxA; ++a)
        if (a < A) io.logits[row * A + a] = lg[a];
    }
    if (ok && io.next_state != nullptr) {  // dense3 head ("+model" actor), not on the acting path
      const float *W3 = w.blob + w.off_w3, *b3 = w.blob + w.off_b3;  // global (L2-resident), see actor_layout
      for (int j = 0; j < D; ++j) {
        float acc = b3[j];
        for (int k = 0; k < kHid; ++k) acc = fmaf(fmaxf(hrow[k * TBP], 0.0f), W3[k * w.Dpad + j], acc);
        io.next_state[row * D + j] = acc;
      }
    }
  }
  __syncthreads();
}

// coalesced write-out of the sampled actions of one tile
template <int N, int TB>
__device__ __forceinline__ void write_actions(const int *s_act, int32_t *act_u, int32_t *act_c, float *onehot,
                                              int64_t env0, int valid, int A0, int A) {
  const int rows = valid * N;
  if (act_u != nullptr)
    for (int r = threadIdx.x; r < rows; r += kActorThreads) act_u[env0 * N + r] = s_act[r * 2];
  if (act_c != nullptr)
    for (int r = threadIdx.x; r < rows; r += kActorThreads) act_c[env0 * N + r] = s_act[r * 2 + 1];
  if (onehot != nullptr)
    for (int i = threadIdx.x; i < rows * A; i += kActorThreads) {
      const int r = i / A, a = i - r * A;
      const bool hot = a < A0 ? (a == s_act[r * 2]) : (a - A0 == s_act[r * 2 + 1]);
      onehot[env0 * N * A + i] = hot ? 1.0f : 0.0f;
    }
}

// ------------------------------------------------------------------------------------------------
// Trainer.get_exploration_action for B envs
// ------------------------------------------------------------------------------------------------
template <int N, int TB, int PAD>
__global__ void __launch_bounds__(kActorThreads, 1) k_actor_forward(ActorDev w, ActorIO io, int64_t ntiles) {
  extern __shared__ __align__(128) float smem_f[];
  ActorSmem<N, TB, PAD> sm;
  sm.carve(smem_f, w.smem_floats, w.D);
  const int tid = threadIdx.x;
  const int ND = N * w.D;
  if (tid == 0) {
    mbar_init(&sm.bars[0], 1);
    mbar_init(&sm.bars[1], 1);
    mbar_fence_init();
    mbar_expect_tx(&sm.bars[0], (uint32_t)(w.smem_floats * sizeof(float)));
    bulk_load(sm.w, w.blob, (uint32_t)(w.smem_floats * sizeof(float)), &sm.bars[0]);
  }
  __syncthreads();
  uint32_t obs_phase = 0;
  bool have_w = false;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t env0 = tile * TB;
    const int valid = (int)((io.B - env0) < TB ? (io.B - env0) : TB);
    if (valid == TB && (reinterpret_cast<uintptr_t>(io.obs) & 15) == 0) {  // one TMA bulk copy of the tile
      if (tid == 0) {
        mbar_expect_tx(&sm.bars[1], (uint32_t)(TB * ND * sizeof(float)));
        bulk_load(sm.obs, io.obs + env0 * ND, (uint32_t)(TB * ND * sizeof(float)), &sm.bars[1]);
      }
      mbar_wait(&sm.bars[1], obs_phase);
      obs_phase ^= 1;
    } else {
      for (int i = tid; i < TB * ND; i += kActorThreads) sm.obs[i] = i < valid * ND ? io.obs[env0 * ND + i] : 0.0f;
      __syncthreads();
    }
    if (!have_w) {
      mbar_wait(&sm.bars[0], 0);
      have_w = true;
    }
    actor_tile<N, TB, PAD>(w, sm, io, env0, valid, io.step);
    write_actions<N, TB>(sm.act, io.act_u, io.act_c, io.onehot, env0, valid, w.A0, w.A);
    __syncthreads();  // sm.obs / sm.act are rewritten by the next tile
  }
}

// ------------------------------------------------------------------------------------------------
// dense3 head of the "+model" actor on top of the tensor-core forward: next_state[row][j] = b3[j] + sum_k
// relu(hcat)[row][k] W3[k][j] (ac_network_model_multi_gumbel.py:49,65).  64 x D MACs per row - HBM-bound on reading
// hcat (256 B per row), so a plain FFMA kernel.  A CTA stages 128 rows of relu(hcat) (32 KB, coalesced float4 loads)
// and the head's weights in shared memory; thread (row pair = tid / 4, quarter = tid % 4) then produces outputs
// quarter, quarter + 4, ... of its two rows: a row's 64 inputs are broadcast reads shared by four threads, the weights
// are re-laid out so that a thread's DQ weights of one k are contiguous and feed 2 x DQ FMAs.  The tensor-core path
// only takes D <= 32 (tc_layout), so DQ <= 8.
// ------------------------------------------------------------------------------------------------
constexpr int kD3Rows2 = 128;
template <int DQ>
__global__ void __launch_bounds__(256) k_dense3x2(ActorDev w, const float *__restrict__ hcat, int64_t rows,
                                                  float *__restrict__ next_state) {
  __shared__ __align__(16) float sh[kD3Rows2][kHid + 4];  // +4: rows start in different banks
  constexpr int DQP = (DQ + 3) / 4 * 4;
  __shared__ __align__(16) float sw3[kHid * 4 * DQP + 4 * DQP];
  const int D = w.D, Dpad = w.Dpad;
  const float *W3 = w.blob + w.off_w3, *b3 = w.blob + w.off_b3;
  for (int i = threadIdx.x; i < kHid * 4 * DQP; i += 256) {
    const int k = i / (4 * DQP), rem = i - k * 4 * DQP, q = rem / DQP, jj = rem - q * DQP, j = q + 4 * jj;
    sw3[i] = (jj < DQ && j < D) ? W3[k * Dpad + j] : 0.0f;
  }
  for (int i = threadIdx.x; i < 4 * DQP; i += 256) {
    const int q = i / DQP, jj = i - q * DQP, j = q + 4 * jj;
    sw3[kHid * 4 * DQP + i] = (jj < DQ && j < D) ? b3[j] : 0.0f;
  }
  const int r = (threadIdx.x >> 2) * 2, qd = threadIdx.x & 3;  // rows r, r + 1 of the tile; outputs qd, qd + 4, ...
  for (int64_t row0 = (int64_t)blockIdx.x * kD3Rows2; row0 < rows; row0 += (int64_t)gridDim.x * kD3Rows2) {
    __syncthreads();  // weights staged / the previous tile is consumed
    for (int i = threadIdx.x; i < kD3Rows2 * (kHid / 4); i += 256) {
      const int rr = i / (kHid / 4), c4 = i - rr * (kHid / 4);
      const float4 v = row0 + rr < rows ? reinterpret_cast<const float4 *>(hcat + (row0 + rr) * kHid)[c4]
                                        : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
      *reinterpret_cast<float4 *>(&sh[rr][4 * c4]) = v;
    }
    __syncthreads();
    float acc[2][DQP];
#pragma unroll
    for (int jj = 0; jj < DQP; ++jj) acc[0][jj] = acc[1][jj] = sw3[kHid * 4 * DQP + qd * DQP + jj];
#pragma unroll 2
    for (int k0 = 0; k0 < kHid; k0 += 4) {
      const float4 ha = *reinterpret_cast<const float4 *>(&sh[r][k0]), hb = *reinterpret_cast<const float4 *>(&sh[r + 1][k0]);
      const float hk[2][4] = {{ha.x, ha.y, ha.z, ha.w}, {hb.x, hb.y, hb.z, hb.w}};
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        const float4 *wk = reinterpret_cast<const float4 *>(sw3 + ((k0 + kk) * 4 + qd) * DQP);
#pragma unroll
        for (int v = 0; v < DQP / 4; ++v) {
          const float4 w4 = wk[v];
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            acc[u][4 * v] = fmaf(hk[u][kk], w4.x, acc[u][4 * v]);
            if (4 * v + 1 < DQ) acc[u][4 * v + 1] = fmaf(hk[u][kk], w4.y, acc[u][4 * v + 1]);
            if (4 * v + 2 < DQ) acc[u][4 * v + 2] = fmaf(hk[u][kk], w4.z, acc[u][4 * v + 2]);
            if (4 * v + 3 < DQ) acc[u][4 * v + 3] = fmaf(hk[u][kk], w4.w, acc[u][4 * v + 3]);
          }
        }
      }
    }
#pragma unroll
    for (int u = 0; u < 2; ++u)
      if (row0 + r + u < rows) {
#pragma unroll
        for (int jj = 0; jj < DQ; ++jj)
          if (qd + 4 * jj < D) next_state[(row0 + r + u) * D + qd + 4 * jj] = acc[u][jj];
      }
  }
}

cudaError_t launch_dense3(const ActorDev &w, const float *hcat, int64_t rows, float *next_state, cudaStream_t st) {
  if (rows <= 0) return cudaSuccess;
  const int64_t nsm = sm_count(current_device());
  const int64_t blocks2 = (rows + kD3Rows2 - 1) / kD3Rows2;
  const unsigned grid2 = (unsigned)(blocks2 < nsm * 5 ? blocks2 : nsm * 5);
  switch ((w.D + 3) / 4) {
#define D3X(Q) case Q: k_dense3x2<Q><<<grid2, 256, 0, st>>>(w, hcat, rows, next_state); break;
    D3X(1) D3X(2) D3X(3) D3X(4) D3X(5) D3X(6) D3X(7) D3X(8)
#undef D3X
    default: return cudaErrorInvalidValue;  // D > 32: no tensor-core forward feeds this head
  }
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// launch
// ------------------------------------------------------------------------------------------------
bool actor_supported(int N) { return N >= 1 && N <= 12; }  // any team size make_env(n=...) is asked for, up to 12
bool rollout_supported(int scenario, int N) { return env_supported(scenario, N); }

template <int N, int TB, int PAD>
static cudaError_t launch_actor_t(const ActorDev &w, const ActorIO &io, cudaStream_t st) {
  const int dev = current_device();
  const size_t smem = ActorSmem<N, TB, PAD>::bytes(w.smem_floats, w.D);
  cudaError_t e = ensure_smem<k_actor_forward<N, TB, PAD>>(smem, dev);
  if (e != cudaSuccess) return e;
  const int64_t ntiles = (io.B + TB - 1) / TB;
  const int nsm = sm_count(dev);
  const int grid = (int)(ntiles < nsm ? ntiles : nsm);
  k_actor_forward<N, TB, PAD><<<grid, kActorThreads, smem, st>>>(w, io, ntiles);
  return cudaGetLastError();
}

cudaError_t launch_actor_forward(const ActorDev &w, const ActorIO &io, cudaStream_t st) {
  switch (io.N) {
    case 1: return launch_actor_t<1, 64, 4>(w, io, st);
    case 2: return launch_actor_t<2, 64, 4>(w, io, st);
    case 3: return launch_actor_t<3, 64, 4>(w, io, st);
    case 4: return launch_actor_t<4, 32, 4>(w, io, st);
    case 5: return launch_actor_t<5, 32, 4>(w, io, st);
    case 6: return launch_actor_t<6, 32, 0>(w, io, st);
    case 7: return launch_actor_t<7, 16, 0>(w, io, st);
    case 8: return launch_actor_t<8, 16, 0>(w, io, st);
    case 9: return launch_actor_t<9, 16, 0>(w, io, st);
    case 10: return launch_actor_t<10, 16, 0>(w, io, st);
    case 11: return launch_actor_t<11, 16, 0>(w, io, st);
    case 12: return launch_actor_t<12, 16, 0>(w, io, st);
    default: return cudaErrorInvalidValue;
  }
}

}  // namespace mpe
