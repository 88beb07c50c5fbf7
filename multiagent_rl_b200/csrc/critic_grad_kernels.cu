// Critic backward: gradients of k_critic_forward's function (critic_kernels.cu) with respect to obs, action and every
// weight tensor, for both reference critics (relu after the attention and one head, or no relu and two heads).
//
// Reference rows: rls/model/ac_network_multi_gumbel.py:70-148 and ac_network_model_multi_gumbel.py:69-143,
// differentiated by Trainer.optimize() (rls/agent/multiagent/ddpg_gumbel_fix.py:131-219): the TD loss through the
// weights, the actor loss through the action.
//
// Three launches, all fp32 FFMA, no floating-point atomics, every sum in an order fixed by the shapes alone:
//   1. k_critic_backward - one warp per sample.  Recomputes the forward from obs, action and the packed weight image
//      with the forward kernel's expressions and accumulation order (so relu masks and attention weights are the
//      forward's), keeping each step's gate activations and cell state in the workspace; then the heads, attention and
//      softmax backward and BPTT over the agent axis.  Writes dobs / daction and, per (sample, agent) row, what the
//      weight gradients are sums of: dgates [256], dz1 [64], x [64], h_{t-1} [64], in [Din]; per sample the heads'
//      input n [64].
//   2. k_grad_partial - the weight gradients as sums over rows (dW_ih = sum dgates^T x, ...), each row range
//      of a fixed chunking summed by one CTA into its own slot of the workspace (grad_reduce.cu, shared with the
//      actor's backward).
//   3. k_grad_sum - the chunk partials summed in chunk order into the caller's tensors.
// Weight gradients cannot be accumulated next to the 151 KB weight image in shared memory, and a warp's registers do
// not hold them either: hence the workspace and the reductions.  One sample per warp (the forward runs four): the
// backward's register arrays leave no room for more, and 148 x 8 warps take B = 1,024 samples in one wave.
#include <cmath>

#include "common.cuh"
#include "critic_launch.h"
#include "grad_reduce.h"
#include "launch.h"

namespace mpe {

namespace {

constexpr int kGradThreads = 256;
constexpr int kGradWarps = kGradThreads / 32;
constexpr int kG = 4 * kCriticH;  // 256 gate rows
// per-row record of the workspace (floats): gate activations, overwritten by dgates (reference row order
// gate * 64 + unit); c_t, overwritten by dz1; x_t = relu(dense1); h_{t-1}; the input row cat(obs, action)
constexpr int kRec = 512, kRecC = 256, kRecX = 320, kRecHp = 384, kRecIn = 448;

__device__ __forceinline__ float sigmoid_acc(float x) { return 1.0f / (1.0f + expf(-x)); }
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

}  // namespace

struct GradWarpSmem {
  float in[kCriticMaxIn];
  float x[kCriticH];
  float h[kCriticH];
  float dz[kCriticH];
  float dg[kG];  // dgates in the weight image's column order: col = lane * 8 + gate * 2 + (unit >= 32)
};

__global__ void __launch_bounds__(kGradThreads, 1)
    k_critic_backward(CriticDev w, const float *__restrict__ obs, const float *__restrict__ action, int64_t B, int N,
                      const float *__restrict__ dq, const float *__restrict__ dr, float *__restrict__ dobs,
                      float *__restrict__ daction, float *__restrict__ rec, float *__restrict__ nrec) {
  extern __shared__ __align__(128) float smem_f[];
  float *sw = smem_f;
  GradWarpSmem *ws = reinterpret_cast<GradWarpSmem *>(sw + w.blob_floats);
  uint64_t *bar = reinterpret_cast<uint64_t *>(ws + kGradWarps);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    mbar_init(bar, 1);
    mbar_fence_init();
    mbar_expect_tx(bar, (uint32_t)(w.blob_floats * sizeof(float)));
    bulk_load(sw, w.blob, (uint32_t)(w.blob_floats * sizeof(float)), bar);
  }
  __syncthreads();
  mbar_wait(bar, 0);
  GradWarpSmem &s = ws[warp];
  const float *Wih = sw + w.off_wih, *Whh = sw + w.off_whh, *bg = sw + w.off_bg + lane * 8;
  const float *W1 = sw + w.off_w1, *b1 = sw + w.off_b1, *W2 = sw + w.off_w2, *W3 = sw + w.off_w3;
  const int D = w.D, A = w.A, Din = w.Din;
  for (int64_t b = (int64_t)blockIdx.x * kGradWarps + warp; b < B; b += (int64_t)gridDim.x * kGradWarps) {
    // ---- forward, as k_critic_forward computes it for one sample
    float c0 = 0.0f, c1 = 0.0f, h0 = 0.0f, h1 = 0.0f;
    float o0[kCriticMaxAgents], o1[kCriticMaxAgents];
    s.h[lane] = 0.0f; s.h[lane + 32] = 0.0f;
#pragma unroll
    for (int t = 0; t < kCriticMaxAgents; ++t) {
      if (t < N) {
        const int64_t row = b * N + t;
        float *r = rec + row * kRec;
        __syncwarp();
        for (int k = lane; k < Din; k += 32) {
          const float v = k < D ? obs[row * D + k] : action[row * A + (k - D)];
          s.in[k] = v;
          r[kRecIn + k] = v;
        }
        __syncwarp();
        float a0 = b1[lane], a1 = b1[lane + 32];
        for (int k = 0; k < Din; ++k) {
          const float xk = s.in[k];
          a0 = fmaf(xk, W1[k * kCriticH + lane], a0);
          a1 = fmaf(xk, W1[k * kCriticH + lane + 32], a1);
        }
        const float x0 = fmaxf(a0, 0.0f), x1 = fmaxf(a1, 0.0f);
        s.x[lane] = x0; s.x[lane + 32] = x1;
        r[kRecX + lane] = x0; r[kRecX + lane + 32] = x1;
        r[kRecHp + lane] = h0; r[kRecHp + lane + 32] = h1;
        __syncwarp();
        float acc[8];
        {
          const float4 bu = *reinterpret_cast<const float4 *>(bg), bv = *reinterpret_cast<const float4 *>(bg + 4);
          acc[0] = bu.x; acc[1] = bu.y; acc[2] = bu.z; acc[3] = bu.w;
          acc[4] = bv.x; acc[5] = bv.y; acc[6] = bv.z; acc[7] = bv.w;
        }
#pragma unroll 2
        for (int k = 0; k < kCriticH; ++k) {
          const float *wi = Wih + k * kG + lane * 8, *wh = Whh + k * kG + lane * 8;
          const float4 iu = *reinterpret_cast<const float4 *>(wi), iv = *reinterpret_cast<const float4 *>(wi + 4);
          const float4 hu = *reinterpret_cast<const float4 *>(wh), hv = *reinterpret_cast<const float4 *>(wh + 4);
          const float xk = s.x[k], hk = s.h[k];
          acc[0] = fmaf(xk, iu.x, acc[0]); acc[1] = fmaf(xk, iu.y, acc[1]);
          acc[2] = fmaf(xk, iu.z, acc[2]); acc[3] = fmaf(xk, iu.w, acc[3]);
          acc[4] = fmaf(xk, iv.x, acc[4]); acc[5] = fmaf(xk, iv.y, acc[5]);
          acc[6] = fmaf(xk, iv.z, acc[6]); acc[7] = fmaf(xk, iv.w, acc[7]);
          acc[0] = fmaf(hk, hu.x, acc[0]); acc[1] = fmaf(hk, hu.y, acc[1]);
          acc[2] = fmaf(hk, hu.z, acc[2]); acc[3] = fmaf(hk, hu.w, acc[3]);
          acc[4] = fmaf(hk, hv.x, acc[4]); acc[5] = fmaf(hk, hv.y, acc[5]);
          acc[6] = fmaf(hk, hv.z, acc[6]); acc[7] = fmaf(hk, hv.w, acc[7]);
        }
        __syncwarp();  // every lane has read h_{t-1}
        const float i0 = sigmoid_acc(acc[0]), i1 = sigmoid_acc(acc[1]), f0 = sigmoid_acc(acc[2]), f1 = sigmoid_acc(acc[3]);
        const float g0 = tanhf(acc[4]), g1 = tanhf(acc[5]), og0 = sigmoid_acc(acc[6]), og1 = sigmoid_acc(acc[7]);
        c0 = f0 * c0 + i0 * g0;
        c1 = f1 * c1 + i1 * g1;
        h0 = og0 * tanhf(c0);
        h1 = og1 * tanhf(c1);
        s.h[lane] = h0; s.h[lane + 32] = h1;
        o0[t] = h0; o1[t] = h1;
        r[lane] = i0; r[lane + 32] = i1; r[64 + lane] = f0; r[96 + lane] = f1;
        r[128 + lane] = g0; r[160 + lane] = g1; r[192 + lane] = og0; r[224 + lane] = og1;
        r[kRecC + lane] = c0; r[kRecC + lane + 32] = c1;
      }
    }
    __syncwarp();
    // attention_net (:103-110): scores = <output_t, h_N>, softmax over the agent axis, weighted sum of the outputs
    float att[kCriticMaxAgents];
    float mx = -INFINITY;
#pragma unroll
    for (int t = 0; t < kCriticMaxAgents; ++t)
      if (t < N) {
        att[t] = warp_sum(o0[t] * h0 + o1[t] * h1);
        mx = fmaxf(mx, att[t]);
      }
    float den = 0.0f;
#pragma unroll
    for (int t = 0; t < kCriticMaxAgents; ++t)
      if (t < N) { att[t] = expf(att[t] - mx); den += att[t]; }
    float n0 = 0.0f, n1 = 0.0f;
#pragma unroll
    for (int t = 0; t < kCriticMaxAgents; ++t)
      if (t < N) {
        att[t] = att[t] / den;
        n0 = fmaf(o0[t], att[t], n0);
        n1 = fmaf(o1[t], att[t], n1);
      }
    nrec[b * kCriticH + lane] = w.relu_attn ? fmaxf(n0, 0.0f) : n0;
    nrec[b * kCriticH + lane + 32] = w.relu_attn ? fmaxf(n1, 0.0f) : n1;

    // ---- heads: dn = dense2^T dq (+ dense3^T dr), through the relu where its output is > 0
    float dn0 = 0.0f, dn1 = 0.0f;
    for (int o = 0; o < w.out; ++o) {
      const float gq = dq[b * w.out + o];
      dn0 = fmaf(gq, W2[lane * kCriticMaxOut + o], dn0);
      dn1 = fmaf(gq, W2[(lane + 32) * kCriticMaxOut + o], dn1);
      if (dr != nullptr) {
        const float gr = dr[b * w.out + o];
        dn0 = fmaf(gr, W3[lane * kCriticMaxOut + o], dn0);
        dn1 = fmaf(gr, W3[(lane + 32) * kCriticMaxOut + o], dn1);
      }
    }
    if (w.relu_attn) {
      dn0 = n0 > 0.0f ? dn0 : 0.0f;
      dn1 = n1 > 0.0f ? dn1 : 0.0f;
    }
    // ---- attention: da_t = <o_t, dn>, softmax backward ds = a (da - sum a da); h_N gets sum_t ds_t o_t as the query
    float ds[kCriticMaxAgents];
    float ada = 0.0f;
#pragma unroll
    for (int t = 0; t < kCriticMaxAgents; ++t)
      if (t < N) {
        ds[t] = warp_sum(o0[t] * dn0 + o1[t] * dn1);
        ada = fmaf(att[t], ds[t], ada);
      }
    float dq0 = 0.0f, dq1 = 0.0f;
#pragma unroll
    for (int t = 0; t < kCriticMaxAgents; ++t)
      if (t < N) {
        ds[t] = att[t] * (ds[t] - ada);
        dq0 = fmaf(ds[t], o0[t], dq0);
        dq1 = fmaf(ds[t], o1[t], dq1);
      }

    // ---- BPTT over the agent axis.  d o_t = a_t dn + ds_t h_N (the keys), plus the query's gradient at t = N - 1
    float gh0 = 0.0f, gh1 = 0.0f, dc0 = 0.0f, dc1 = 0.0f;  // gradient reaching h_t / c_t from step t + 1
#pragma unroll
    for (int t = kCriticMaxAgents - 1; t >= 0; --t) {
      if (t < N) {
        const int64_t row = b * N + t;
        float *r = rec + row * kRec;
        float e0 = fmaf(att[t], dn0, fmaf(ds[t], h0, gh0)), e1 = fmaf(att[t], dn1, fmaf(ds[t], h1, gh1));
        if (t == N - 1) { e0 += dq0; e1 += dq1; }
        const float i0 = r[lane], i1 = r[lane + 32], f0 = r[64 + lane], f1 = r[96 + lane];
        const float g0 = r[128 + lane], g1 = r[160 + lane], og0 = r[192 + lane], og1 = r[224 + lane];
        const float ct0 = r[kRecC + lane], ct1 = r[kRecC + lane + 32];
        const float cp0 = t > 0 ? r[kRecC - kRec + lane] : 0.0f, cp1 = t > 0 ? r[kRecC - kRec + lane + 32] : 0.0f;
        const float tc0 = tanhf(ct0), tc1 = tanhf(ct1);
        const float do0 = e0 * tc0 * (og0 * (1.0f - og0)), do1 = e1 * tc1 * (og1 * (1.0f - og1));
        dc0 = fmaf(e0 * og0, 1.0f - tc0 * tc0, dc0);
        dc1 = fmaf(e1 * og1, 1.0f - tc1 * tc1, dc1);
        const float di0 = dc0 * g0 * (i0 * (1.0f - i0)), di1 = dc1 * g1 * (i1 * (1.0f - i1));
        const float dg0 = dc0 * i0 * (1.0f - g0 * g0), dg1 = dc1 * i1 * (1.0f - g1 * g1);
        const float df0 = dc0 * cp0 * (f0 * (1.0f - f0)), df1 = dc1 * cp1 * (f1 * (1.0f - f1));
        dc0 *= f0;
        dc1 *= f1;
        r[lane] = di0; r[lane + 32] = di1; r[64 + lane] = df0; r[96 + lane] = df1;
        r[128 + lane] = dg0; r[160 + lane] = dg1; r[192 + lane] = do0; r[224 + lane] = do1;
        *reinterpret_cast<float4 *>(s.dg + lane * 8) = make_float4(di0, di1, df0, df1);
        *reinterpret_cast<float4 *>(s.dg + lane * 8 + 4) = make_float4(dg0, dg1, do0, do1);
        __syncwarp();
        // dx = W_ih^T dgates and dh_{t-1} = W_hh^T dgates at k = lane, lane + 32: row k of an image holds the 256
        // gate columns of input k; each lane starts at its own column quad, so the warp's loads hit distinct banks
        float dx0 = 0.0f, dx1 = 0.0f, dp0 = 0.0f, dp1 = 0.0f;
#pragma unroll 4
        for (int c = 0; c < kG / 4; ++c) {
          const int q = ((c + lane) & (kG / 4 - 1)) * 4;
          const float4 d = *reinterpret_cast<const float4 *>(s.dg + q);
          const float4 a = *reinterpret_cast<const float4 *>(Wih + lane * kG + q);
          const float4 a2 = *reinterpret_cast<const float4 *>(Wih + (lane + 32) * kG + q);
          const float4 e = *reinterpret_cast<const float4 *>(Whh + lane * kG + q);
          const float4 e2 = *reinterpret_cast<const float4 *>(Whh + (lane + 32) * kG + q);
          dx0 = fmaf(a.x, d.x, dx0); dx0 = fmaf(a.y, d.y, dx0); dx0 = fmaf(a.z, d.z, dx0); dx0 = fmaf(a.w, d.w, dx0);
          dx1 = fmaf(a2.x, d.x, dx1); dx1 = fmaf(a2.y, d.y, dx1); dx1 = fmaf(a2.z, d.z, dx1); dx1 = fmaf(a2.w, d.w, dx1);
          dp0 = fmaf(e.x, d.x, dp0); dp0 = fmaf(e.y, d.y, dp0); dp0 = fmaf(e.z, d.z, dp0); dp0 = fmaf(e.w, d.w, dp0);
          dp1 = fmaf(e2.x, d.x, dp1); dp1 = fmaf(e2.y, d.y, dp1); dp1 = fmaf(e2.z, d.z, dp1); dp1 = fmaf(e2.w, d.w, dp1);
        }
        gh0 = dp0; gh1 = dp1;
        // relu(dense1): the gradient passes where x = relu(z1) > 0
        const float dz0 = r[kRecX + lane] > 0.0f ? dx0 : 0.0f, dz1 = r[kRecX + lane + 32] > 0.0f ? dx1 : 0.0f;
        r[kRecC + lane] = dz0; r[kRecC + lane + 32] = dz1;  // c_t is not read again
        if (dobs != nullptr || daction != nullptr) {
          s.dz[lane] = dz0; s.dz[lane + 32] = dz1;
          __syncwarp();
          // d in = dense1^T dz1 at k = lane, lane + 32 (row k of the dense1 image holds its 64 units)
          for (int k = lane; k < Din; k += 32) {
            float v = 0.0f;
#pragma unroll 4
            for (int c = 0; c < kCriticH / 4; ++c) {
              const int q = ((c + lane) & (kCriticH / 4 - 1)) * 4;
              const float4 z = *reinterpret_cast<const float4 *>(s.dz + q);
              const float4 wv = *reinterpret_cast<const float4 *>(W1 + k * kCriticH + q);
              v = fmaf(wv.x, z.x, v); v = fmaf(wv.y, z.y, v); v = fmaf(wv.z, z.z, v); v = fmaf(wv.w, z.w, v);
            }
            if (k < D) {
              if (dobs != nullptr) dobs[row * D + k] = v;
            } else if (daction != nullptr) {
              daction[row * A + (k - D)] = v;
            }
          }
        }
        __syncwarp();  // s.dg / s.dz are rewritten by the next step
      }
    }
  }
}

namespace {

// Where everything lives: the workspace is [rows][kRec] records, [B][64] heads' inputs, [nchunk][nout] partials;
// the partial vector holds W_ih, W_hh, gate bias, dense1 w / b, dense2 w / b, dense3 w / b.
struct GradPlan {
  int64_t rows, off_n, off_part, floats;
  int nchunk, nout;
  int o_wih, o_whh, o_bg, o_w1, o_b1, o_w2, o_b2, o_w3, o_b3;
};

GradPlan grad_plan(const CriticDev &w, int64_t B, int N) {
  GradPlan p;
  p.rows = B * N;
  p.nchunk = grad_chunks(p.rows);
  int off = 0;
  p.o_wih = off; off += kG * kCriticH;
  p.o_whh = off; off += kG * kCriticH;
  p.o_bg = off; off += kG;
  p.o_w1 = off; off += kCriticH * w.Din;
  p.o_b1 = off; off += kCriticH;
  p.o_w2 = off; off += w.out * kCriticH;
  p.o_b2 = off; off += w.out;
  p.o_w3 = off; off += w.out * kCriticH;
  p.o_b3 = off; off += w.out;
  p.nout = (off + 63) / 64 * 64;
  p.off_n = p.rows * kRec;
  p.off_part = p.off_n + B * kCriticH;
  p.floats = p.off_part + (int64_t)p.nchunk * p.nout;
  return p;
}

}  // namespace

int64_t critic_backward_bytes(const CriticDev &w, int64_t B, int N) {
  return B <= 0 ? 0 : grad_plan(w, B, N).floats * (int64_t)sizeof(float);
}

cudaError_t launch_critic_backward(const CriticDev &w, const float *obs, const float *action, int64_t B, int N,
                                   const float *dq, const float *dr, float *dobs, float *daction,
                                   const CriticGrads &g, void *workspace, cudaStream_t st) {
  if (B <= 0) return cudaSuccess;
  if (N < 1 || N > kCriticMaxAgents) return cudaErrorInvalidValue;
  const GradPlan p = grad_plan(w, B, N);
  float *ws = static_cast<float *>(workspace);
  const int dev = current_device();
  const size_t smem = w.blob_floats * sizeof(float) + kGradWarps * sizeof(GradWarpSmem) + 64;
  cudaError_t e = ensure_smem<k_critic_backward>(smem, dev);
  if (e != cudaSuccess) return e;
  const int nsm = sm_count(dev);
  const int64_t want = (B + kGradWarps - 1) / kGradWarps;
  k_critic_backward<<<(int)(want < nsm ? want : nsm), kGradThreads, smem, st>>>(w, obs, action, B, N, dq, dr, dobs,
                                                                               daction, ws, ws + p.off_n);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;

  GradSegs segs = {};
  auto seg = [&](float *dst, int src, int n) {
    if (dst != nullptr) segs.s[segs.nseg++] = GradSeg{dst, src, n};
  };
  const int H = kCriticH, O = w.out;
  seg(g.dense1_w, p.o_w1, H * w.Din);
  seg(g.dense1_b, p.o_b1, H);
  seg(g.w_ih, p.o_wih, kG * H);
  seg(g.w_hh, p.o_whh, kG * H);
  seg(g.b_ih, p.o_bg, kG);
  seg(g.b_hh, p.o_bg, kG);
  seg(g.dense2_w, p.o_w2, O * H);
  seg(g.dense2_b, p.o_b2, O);
  seg(g.dense3_w, dr != nullptr ? p.o_w3 : -1, O * H);
  seg(g.dense3_b, dr != nullptr ? p.o_b3 : -1, O);
  if (segs.nseg == 0) return cudaSuccess;

  const float *rec = ws;
  GradTiles tiles = {};
  int nt = 0;
  for (int mt = 0; mt < kG / 64; ++mt) {  // dW_ih = sum dgates^T x (+ the gate bias), dW_hh = sum dgates^T h_{t-1}
    tiles.t[nt++] = GradTile{rec + mt * 64, rec + kRecX, p.rows, kRec, kRec, 64, H, p.o_wih + mt * 64 * H, H, p.o_bg + mt * 64};
    tiles.t[nt++] = GradTile{rec + mt * 64, rec + kRecHp, p.rows, kRec, kRec, 64, H, p.o_whh + mt * 64 * H, H, -1};
  }
  tiles.t[nt++] = GradTile{rec + kRecC, rec + kRecIn, p.rows, kRec, kRec, H, w.Din, p.o_w1, w.Din, p.o_b1};  // dense1
  tiles.t[nt++] = GradTile{dq, ws + p.off_n, B, O, H, O, H, p.o_w2, H, p.o_b2};                          // dense2
  if (dr != nullptr) tiles.t[nt++] = GradTile{dr, ws + p.off_n, B, O, H, O, H, p.o_w3, H, p.o_b3};       // dense3
  tiles.nchunk = p.nchunk;
  tiles.nout = p.nout;
  return launch_grad_reduce(tiles, nt, segs, ws + p.off_part, st);
}

}  // namespace mpe
