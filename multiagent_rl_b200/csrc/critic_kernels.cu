// Critic forward: cat(obs, action) -> relu(dense1) -> LSTM(64) over the agent axis -> dot-product attention with the
// final hidden state -> softmax over agents -> weighted sum (-> relu) -> dense2 (and dense3 for the "+model" critic).
//
// Reference rows: rls/model/ac_network_multi_gumbel.py:70-148 (CriticNetwork.forward :123-148, attention_net :94-121),
// rls/model/ac_network_model_multi_gumbel.py:69-143 (two heads, no relu after the attention), called from
// rls/agent/multiagent/ddpg_gumbel_fix.py:151,159,191 (optimize) and model_ddpg_gumbel_fix.py:155,163,199.
// SURVEY 8f-2: not on the acting path; here so that imagined rollouts / TD targets can stay on the device.
//
// Mapping: one warp per pair of samples (each weight row read from shared memory serves both).  A persistent CTA (8 warps) keeps the packed weights (W_ih, W_hh: 2 x 64 x 256 fp32 =
// 128 KB, plus dense1 / heads) in shared memory, loaded once with a TMA bulk copy.  Lane l owns hidden units l and
// l + 32: its 8 gate pre-activations per step are one 32 B slice of a k-major weight row, x_t / h_{t-1} are broadcast
// reads of the warp's staging row.  All arithmetic fp32 (FFMA), exp / tanh by the accurate libdevice forms.
#include <cmath>

#include "common.cuh"
#include "critic_launch.h"
#include "launch.h"

namespace mpe {

constexpr int kCriticThreads = 256;
constexpr int kCriticWarps = kCriticThreads / 32;
constexpr int kGates = 4 * kCriticH;  // 256

static int round_up4(int x) { return (x + 3) / 4 * 4; }

void critic_layout(int D, int A, int out, bool has_r, bool relu_attn, CriticDev *o) {
  o->D = D; o->A = A; o->Din = D + A; o->out = out; o->has_r = has_r ? 1 : 0; o->relu_attn = relu_attn ? 1 : 0;
  int off = 0;
  o->off_wih = off; off += kCriticH * kGates;
  o->off_whh = off; off += kCriticH * kGates;
  o->off_bg = off; off += kGates;
  o->off_w1 = off; off += round_up4(o->Din * kCriticH);
  o->off_b1 = off; off += kCriticH;
  o->off_w2 = off; off += kCriticH * kCriticMaxOut;
  o->off_b2 = off; off += kCriticMaxOut;
  o->off_w3 = off; off += kCriticH * kCriticMaxOut;
  o->off_b3 = off; off += kCriticMaxOut;
  o->blob_floats = (size_t)((off + 31) / 32 * 32);
}

__device__ __forceinline__ float sigmoid_acc(float x) { return 1.0f / (1.0f + expf(-x)); }
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

constexpr int kCriticR = 4;  // samples per warp and pass: every weight row read from shared memory serves all of them
                             // (1: 1.61 ms, 2: 1.06 ms, 4: 0.90 ms for 65,536 x 3 agent rows; 235 registers, no spills)

// per-warp staging: the input rows, x_t = relu(dense1) and h_{t-1} of the warp's kCriticR samples (every step's output,
// which the attention needs, stays in the registers of the lane that owns the unit)
struct CriticWarpSmem {
  float in[kCriticR][kCriticMaxIn];
  float x[kCriticR][kCriticH];
  float h[kCriticR][kCriticH];
};

__global__ void __launch_bounds__(kCriticThreads, 1)
    k_critic_forward(CriticDev w, const float *__restrict__ obs, const float *__restrict__ action, int64_t B, int N,
                     float *__restrict__ q, float *__restrict__ r) {
  extern __shared__ __align__(128) float smem_f[];
  float *sw = smem_f;
  CriticWarpSmem *ws = reinterpret_cast<CriticWarpSmem *>(sw + w.blob_floats);
  uint64_t *bar = reinterpret_cast<uint64_t *>(ws + kCriticWarps);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    mbar_init(bar, 1);
    mbar_fence_init();
    mbar_expect_tx(bar, (uint32_t)(w.blob_floats * sizeof(float)));
    bulk_load(sw, w.blob, (uint32_t)(w.blob_floats * sizeof(float)), bar);
  }
  __syncthreads();
  mbar_wait(bar, 0);
  CriticWarpSmem &s = ws[warp];
  const float *Wih = sw + w.off_wih + lane * 8, *Whh = sw + w.off_whh + lane * 8, *bg = sw + w.off_bg + lane * 8;
  const float *W1 = sw + w.off_w1, *b1 = sw + w.off_b1;
  const int D = w.D, A = w.A, Din = w.Din;
  const int64_t npass = (B + kCriticR - 1) / kCriticR;
  for (int64_t pass = (int64_t)blockIdx.x * kCriticWarps + warp; pass < npass; pass += (int64_t)gridDim.x * kCriticWarps) {
    int64_t bs[kCriticR];
    bool ok[kCriticR];
#pragma unroll
    for (int u = 0; u < kCriticR; ++u) {
      ok[u] = pass * kCriticR + u < B;
      bs[u] = ok[u] ? pass * kCriticR + u : pass * kCriticR;  // a ragged tail recomputes its first sample, stores nothing
    }
    float c0[kCriticR], c1[kCriticR], h0[kCriticR], h1[kCriticR];
    float o0[kCriticR][kCriticMaxAgents], o1[kCriticR][kCriticMaxAgents];  // outputs of the lane's two units, per step
#pragma unroll
    for (int u = 0; u < kCriticR; ++u) {
      c0[u] = c1[u] = h0[u] = h1[u] = 0.0f;
      s.h[u][lane] = 0.0f; s.h[u][lane + 32] = 0.0f;
    }
#pragma unroll
    for (int t = 0; t < kCriticMaxAgents; ++t) {
      if (t < N) {
        // obs_act = cat(obs, action) (ac_network_multi_gumbel.py:131-134)
        __syncwarp();
#pragma unroll
        for (int u = 0; u < kCriticR; ++u)
          for (int k = lane; k < Din; k += 32)
            s.in[u][k] = k < D ? obs[(bs[u] * N + t) * D + k] : action[(bs[u] * N + t) * A + (k - D)];
        __syncwarp();
        // relu(dense1): lane computes outputs lane and lane + 32
        float a0[kCriticR], a1[kCriticR];
#pragma unroll
        for (int u = 0; u < kCriticR; ++u) { a0[u] = b1[lane]; a1[u] = b1[lane + 32]; }
        for (int k = 0; k < Din; ++k) {
          const float wa = W1[k * kCriticH + lane], wb = W1[k * kCriticH + lane + 32];
#pragma unroll
          for (int u = 0; u < kCriticR; ++u) {
            const float xk = s.in[u][k];
            a0[u] = fmaf(xk, wa, a0[u]);
            a1[u] = fmaf(xk, wb, a1[u]);
          }
        }
#pragma unroll
        for (int u = 0; u < kCriticR; ++u) { s.x[u][lane] = fmaxf(a0[u], 0.0f); s.x[u][lane + 32] = fmaxf(a1[u], 0.0f); }
        __syncwarp();
        // gates = b + W_ih x_t + W_hh h_{t-1}; packed columns [i0 i1 f0 f1 g0 g1 o0 o1] of units (lane, lane + 32)
        float acc[kCriticR][8];
        {
          const float4 bu = *reinterpret_cast<const float4 *>(bg), bv = *reinterpret_cast<const float4 *>(bg + 4);
#pragma unroll
          for (int u = 0; u < kCriticR; ++u) {
            acc[u][0] = bu.x; acc[u][1] = bu.y; acc[u][2] = bu.z; acc[u][3] = bu.w;
            acc[u][4] = bv.x; acc[u][5] = bv.y; acc[u][6] = bv.z; acc[u][7] = bv.w;
          }
        }
#pragma unroll 2
        for (int k = 0; k < kCriticH; ++k) {
          const float4 iu = *reinterpret_cast<const float4 *>(Wih + k * kGates), iv = *reinterpret_cast<const float4 *>(Wih + k * kGates + 4);
          const float4 hu = *reinterpret_cast<const float4 *>(Whh + k * kGates), hv = *reinterpret_cast<const float4 *>(Whh + k * kGates + 4);
#pragma unroll
          for (int u = 0; u < kCriticR; ++u) {
            const float xk = s.x[u][k], hk = s.h[u][k];
            acc[u][0] = fmaf(xk, iu.x, acc[u][0]); acc[u][1] = fmaf(xk, iu.y, acc[u][1]);
            acc[u][2] = fmaf(xk, iu.z, acc[u][2]); acc[u][3] = fmaf(xk, iu.w, acc[u][3]);
            acc[u][4] = fmaf(xk, iv.x, acc[u][4]); acc[u][5] = fmaf(xk, iv.y, acc[u][5]);
            acc[u][6] = fmaf(xk, iv.z, acc[u][6]); acc[u][7] = fmaf(xk, iv.w, acc[u][7]);
            acc[u][0] = fmaf(hk, hu.x, acc[u][0]); acc[u][1] = fmaf(hk, hu.y, acc[u][1]);
            acc[u][2] = fmaf(hk, hu.z, acc[u][2]); acc[u][3] = fmaf(hk, hu.w, acc[u][3]);
            acc[u][4] = fmaf(hk, hv.x, acc[u][4]); acc[u][5] = fmaf(hk, hv.y, acc[u][5]);
            acc[u][6] = fmaf(hk, hv.z, acc[u][6]); acc[u][7] = fmaf(hk, hv.w, acc[u][7]);
          }
        }
        __syncwarp();  // every lane has read h_{t-1}
#pragma unroll
        for (int u = 0; u < kCriticR; ++u) {
          c0[u] = sigmoid_acc(acc[u][2]) * c0[u] + sigmoid_acc(acc[u][0]) * tanhf(acc[u][4]);
          c1[u] = sigmoid_acc(acc[u][3]) * c1[u] + sigmoid_acc(acc[u][1]) * tanhf(acc[u][5]);
          h0[u] = sigmoid_acc(acc[u][6]) * tanhf(c0[u]);
          h1[u] = sigmoid_acc(acc[u][7]) * tanhf(c1[u]);
          s.h[u][lane] = h0[u]; s.h[u][lane + 32] = h1[u];
          o0[u][t] = h0[u]; o1[u][t] = h1[u];
        }
      }
    }
    __syncwarp();
    // attention_net (:103-110): scores = <output_t, h_N>, softmax over the agent axis, weighted sum of the outputs
#pragma unroll
    for (int u = 0; u < kCriticR; ++u) {
      float score[kCriticMaxAgents];
      float mx = -INFINITY;
#pragma unroll
      for (int t = 0; t < kCriticMaxAgents; ++t)
        if (t < N) {
          score[t] = warp_sum(o0[u][t] * h0[u] + o1[u][t] * h1[u]);
          mx = fmaxf(mx, score[t]);
        }
      float den = 0.0f;
#pragma unroll
      for (int t = 0; t < kCriticMaxAgents; ++t)
        if (t < N) { score[t] = expf(score[t] - mx); den += score[t]; }
      float n0 = 0.0f, n1 = 0.0f;
#pragma unroll
      for (int t = 0; t < kCriticMaxAgents; ++t)
        if (t < N) {
          const float a = score[t] / den;
          n0 = fmaf(o0[u][t], a, n0);
          n1 = fmaf(o1[u][t], a, n1);
        }
      if (w.relu_attn) { n0 = fmaxf(n0, 0.0f); n1 = fmaxf(n1, 0.0f); }  // ac_network_multi_gumbel.py:141 only
      for (int o = 0; o < w.out; ++o) {
        const float *W2 = sw + w.off_w2;
        const float v = warp_sum(n0 * W2[lane * kCriticMaxOut + o] + n1 * W2[(lane + 32) * kCriticMaxOut + o]);
        if (lane == 0 && ok[u]) q[bs[u] * w.out + o] = v + sw[w.off_b2 + o];
        if (w.has_r && r != nullptr) {
          const float *W3 = sw + w.off_w3;
          const float uu = warp_sum(n0 * W3[lane * kCriticMaxOut + o] + n1 * W3[(lane + 32) * kCriticMaxOut + o]);
          if (lane == 0 && ok[u]) r[bs[u] * w.out + o] = uu + sw[w.off_b3 + o];
        }
      }
    }
  }
}

cudaError_t launch_critic_forward(const CriticDev &w, const float *obs, const float *action, int64_t B, int N, float *q,
                                  float *r, cudaStream_t st) {
  if (B <= 0) return cudaSuccess;
  if (N < 1 || N > kCriticMaxAgents) return cudaErrorInvalidValue;
  const int dev = current_device();
  const size_t smem = w.blob_floats * sizeof(float) + kCriticWarps * sizeof(CriticWarpSmem) + 64;
  cudaError_t e = ensure_smem<k_critic_forward>(smem, dev);
  if (e != cudaSuccess) return e;
  const int nsm = sm_count(dev);
  const int64_t want = ((B + kCriticR - 1) / kCriticR + kCriticWarps - 1) / kCriticWarps;
  const int grid = (int)(want < nsm ? want : nsm);
  k_critic_forward<<<grid, kCriticThreads, smem, st>>>(w, obs, action, B, N, q, r);
  return cudaGetLastError();
}

}  // namespace mpe
