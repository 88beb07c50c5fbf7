// Actor backward: gradients of the function k_actor_forward computes on its fp32 FFMA path (actor_kernels.cu) with
// respect to obs and every weight tensor, for every actor the forward covers (1..12 agents, D <= 64, one or two heads,
// the optional dense3 "+model" head).
//
// Reference rows: rls/model/ac_network_multi_gumbel.py:24-67 and ac_network_model_multi_gumbel.py:23-66,
// differentiated by Trainer.optimize() (rls/agent/multiagent/ddpg_gumbel_fix.py:131-219): the actor loss through the
// weights.
//
// Three launches, all fp32 FFMA, no floating-point atomics, every sum in an order fixed by the shapes alone:
//   1. k_actor_backward - one warp per sample.  Recomputes the forward from obs and the packed weight image with the
//      forward kernel's expressions and accumulation order (dense1 as b1 + sum_k fmaf in k order; the gates as the
//      pre-summed bias, then x over k = 0..63, then h_{s-1} over k = 0..31; actor_cell.cuh's activations), so every
//      relu mask is the forward's.  Lane dir * 16 + ug owns the forward's 8 packed gate columns of units ug and
//      ug + 16 of direction dir: both half-warps step together, the forward direction on agent s and the reverse one
//      on agent N - 1 - s, keeping each step's gate activations and cell state in the workspace.  Then the heads'
//      backward through relu(hcat), BPTT of both directions (the reverse direction's previous state is agent t + 1's),
//      dx = W_ih^T dgates over both directions, the dense1 relu and dobs = W1^T dz1.  Per (sample, agent) row it
//      leaves in the workspace what the weight gradients are sums of: dgates of both directions [256], dz1 [64],
//      x = relu(z1) [64], h_{s-1} of both directions [64], relu(hcat) [64].
//   2. + 3. grad_reduce.cu: the row sums (11 tiles: W_ih and W_hh two each per direction, dense1, both heads in one
//      tile, dense3), chunked and then added in chunk order.
#include <cmath>

#include "actor_cell.cuh"
#include "actor_launch.h"
#include "common.cuh"
#include "grad_reduce.h"
#include "launch.h"

namespace mpe {

namespace {

constexpr int kAgThreads = 256;
constexpr int kAgWarps = kAgThreads / 32;
constexpr int kMaxAgents = 12;
constexpr int kXs = kHid + 1;  // row stride of the per-agent arrays: the two half-warps read different agents' rows
// per-row record of the workspace (floats): gate activations of direction d at d * 128 + gate * 32 + unit (reference
// row order), overwritten by dgates; c_t of direction d at kRecC + d * 32 + unit, overwritten by dz1; x = relu(z1);
// h_{s-1} of direction d at kRecHp + d * 32; relu(hcat)
constexpr int kRec = 512, kRecC = 256, kRecX = 320, kRecHp = 384, kRecH = 448;

struct ActorGradSmem {
  float x[kMaxAgents * kXs];   // relu(dense1) of every agent
  float hd[kMaxAgents * kXs];  // hcat (the BiLSTM output) of every agent, then its gradient through the relu
  float in[kActorMaxD];
  float h[2 * kH];       // h_{s-1} of each direction
  float dg[2 * kGateN];  // dgates of each direction in the weight image's column order ug * 8 + gate * 2 + uu
  float dz[kHid];
};

}  // namespace

__global__ void __launch_bounds__(kAgThreads, 1)
    k_actor_backward(ActorDev w, const float *__restrict__ obs, int64_t B, int N, const float *__restrict__ dlogits,
                     const float *__restrict__ dns, float *__restrict__ dobs, float *__restrict__ rec) {
  extern __shared__ __align__(128) float smem_f[];
  float *sw = smem_f;                            // the forward's staged image (everything but dense3)
  float *w2t = sw + w.smem_floats;               // [A][64]: both heads, transposed
  float *w3t = w2t + kActorMaxA * kHid;          // [D][64]: dense3, transposed ("+model" actor)
  const int nw3 = w.has_model ? w.D * kHid : 0;
  ActorGradSmem *wsm = reinterpret_cast<ActorGradSmem *>(w3t + nw3);
  uint64_t *bar = reinterpret_cast<uint64_t *>(wsm + kAgWarps);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    mbar_init(bar, 1);
    mbar_fence_init();
    mbar_expect_tx(bar, (uint32_t)(w.smem_floats * sizeof(float)));
    bulk_load(sw, w.blob, (uint32_t)(w.smem_floats * sizeof(float)), bar);
  }
  __syncthreads();
  mbar_wait(bar, 0);
  for (int i = tid; i < w.A * kHid; i += kAgThreads) w2t[i] = sw[w.off_w2 + (i % kHid) * w.Apad + i / kHid];
  for (int i = tid; i < nw3; i += kAgThreads) w3t[i] = w.blob[w.off_w3 + (i % kHid) * w.Dpad + i / kHid];
  __syncthreads();

  ActorGradSmem &s = wsm[warp];
  const int D = w.D, A = w.A;
  const int dir = lane >> 4, ug = lane & 15;
  const float *W1 = sw + w.off_w1, *b1 = sw + w.off_b1;
  const float *Wd = sw + w.off_wg[dir];  // this lane's direction: [96][128], rows 0..63 W_ih, 64..95 W_hh
  const float *Wg = Wd + ug * 8;         // ... at this lane's 8 columns
  const float *bg = sw + w.off_bg + dir * kGateN + ug * 8;
  for (int64_t b = (int64_t)blockIdx.x * kAgWarps + warp; b < B; b += (int64_t)gridDim.x * kAgWarps) {
    float *rb = rec + b * N * kRec;
    // ---- dense1, as k_actor_forward computes it: x = relu(b1 + sum_k fmaf(obs_k, W1[k]))
    for (int t = 0; t < N; ++t) {
      float *r = rb + t * kRec;
      __syncwarp();
      for (int k = lane; k < D; k += 32) s.in[k] = obs[(b * N + t) * D + k];
      __syncwarp();
      float a0 = b1[lane], a1 = b1[lane + 32];
      for (int k = 0; k < D; ++k) {
        const float xk = s.in[k];
        a0 = fmaf(xk, W1[k * kHid + lane], a0);
        a1 = fmaf(xk, W1[k * kHid + lane + 32], a1);
      }
      const float x0 = fmaxf(a0, 0.0f), x1 = fmaxf(a1, 0.0f);
      s.x[t * kXs + lane] = x0; s.x[t * kXs + lane + 32] = x1;
      r[kRecX + lane] = x0; r[kRecX + lane + 32] = x1;
    }
    s.h[lane] = 0.0f; s.h[lane + 32] = 0.0f;
    __syncwarp();

    // ---- BiLSTM: step st of direction dir is agent t; the gate sums in the forward's order
    float c0 = 0.0f, c1 = 0.0f;
    for (int st = 0; st < N; ++st) {
      const int t = dir == 0 ? st : N - 1 - st;
      float *r = rb + t * kRec;
      float acc[8];
      {
        const float4 bu = *reinterpret_cast<const float4 *>(bg), bv = *reinterpret_cast<const float4 *>(bg + 4);
        acc[0] = bu.x; acc[1] = bu.y; acc[2] = bu.z; acc[3] = bu.w;
        acc[4] = bv.x; acc[5] = bv.y; acc[6] = bv.z; acc[7] = bv.w;
      }
      const float *xt = s.x + t * kXs;
#pragma unroll 4
      for (int k = 0; k < kHid; ++k) {
        const float4 u = *reinterpret_cast<const float4 *>(Wg + k * kGateN);
        const float4 v = *reinterpret_cast<const float4 *>(Wg + k * kGateN + 4);
        const float xk = xt[k];
        acc[0] = fmaf(xk, u.x, acc[0]); acc[1] = fmaf(xk, u.y, acc[1]);
        acc[2] = fmaf(xk, u.z, acc[2]); acc[3] = fmaf(xk, u.w, acc[3]);
        acc[4] = fmaf(xk, v.x, acc[4]); acc[5] = fmaf(xk, v.y, acc[5]);
        acc[6] = fmaf(xk, v.z, acc[6]); acc[7] = fmaf(xk, v.w, acc[7]);
      }
      const float *hp = s.h + dir * kH;
      if (st > 0) {  // the forward has no h_{-1} term at all
#pragma unroll 4
        for (int k = 0; k < kH; ++k) {
          const float4 u = *reinterpret_cast<const float4 *>(Wg + (kHid + k) * kGateN);
          const float4 v = *reinterpret_cast<const float4 *>(Wg + (kHid + k) * kGateN + 4);
          const float hk = hp[k];
          acc[0] = fmaf(hk, u.x, acc[0]); acc[1] = fmaf(hk, u.y, acc[1]);
          acc[2] = fmaf(hk, u.z, acc[2]); acc[3] = fmaf(hk, u.w, acc[3]);
          acc[4] = fmaf(hk, v.x, acc[4]); acc[5] = fmaf(hk, v.y, acc[5]);
          acc[6] = fmaf(hk, v.z, acc[6]); acc[7] = fmaf(hk, v.w, acc[7]);
        }
      }
      r[kRecHp + dir * kH + ug] = hp[ug];
      r[kRecHp + dir * kH + ug + 16] = hp[ug + 16];
      __syncwarp();  // every lane has read h_{s-1}
      float *rg = r + dir * kGateN;
#pragma unroll
      for (int uu = 0; uu < 2; ++uu) {  // packed columns: [i0 i1 f0 f1 g0 g1 o0 o1] for units (ug, ug + 16)
        const int u = ug + 16 * uu;
        const float ig = sigmoid_f(acc[0 + uu]), fg = sigmoid_f(acc[2 + uu]);
        const float gg = tanh_f(acc[4 + uu]), og = sigmoid_f(acc[6 + uu]);
        float &c = uu ? c1 : c0;
        c = fmaf(fg, c, ig * gg);
        const float h = og * tanh_f(c);
        s.h[dir * kH + u] = h;
        s.hd[t * kXs + dir * kH + u] = h;
        rg[u] = ig; rg[kH + u] = fg; rg[2 * kH + u] = gg; rg[3 * kH + u] = og;
        r[kRecC + dir * kH + u] = c;
      }
      __syncwarp();
    }

    // ---- heads: dhcat = dense2^T dlogits (+ dense3^T dnext_state), through the relu where hcat > 0
    for (int t = 0; t < N; ++t) {
      const int64_t row = b * N + t;
      float *r = rb + t * kRec;
      const float gl = lane < A ? dlogits[row * A + lane] : 0.0f;
      float d0 = 0.0f, d1 = 0.0f;
      for (int a = 0; a < A; ++a) {
        const float g = __shfl_sync(0xffffffffu, gl, a);
        d0 = fmaf(g, w2t[a * kHid + lane], d0);
        d1 = fmaf(g, w2t[a * kHid + lane + 32], d1);
      }
      if (dns != nullptr) {
        const float n0 = lane < D ? dns[row * D + lane] : 0.0f, n1 = lane + 32 < D ? dns[row * D + lane + 32] : 0.0f;
        for (int j = 0; j < D; ++j) {
          const float g = __shfl_sync(0xffffffffu, j < 32 ? n0 : n1, j & 31);
          d0 = fmaf(g, w3t[j * kHid + lane], d0);
          d1 = fmaf(g, w3t[j * kHid + lane + 32], d1);
        }
      }
      float *hd = s.hd + t * kXs;
      const float h0 = hd[lane], h1 = hd[lane + 32];
      r[kRecH + lane] = fmaxf(h0, 0.0f); r[kRecH + lane + 32] = fmaxf(h1, 0.0f);
      hd[lane] = h0 > 0.0f ? d0 : 0.0f;
      hd[lane + 32] = h1 > 0.0f ? d1 : 0.0f;
    }
    __syncwarp();

    // ---- BPTT, both directions at once from their last step; gh = gradient reaching h_s from step s + 1
    float gh0 = 0.0f, gh1 = 0.0f, dc0 = 0.0f, dc1 = 0.0f;
    for (int st = N - 1; st >= 0; --st) {
      const int t = dir == 0 ? st : N - 1 - st;
      float *r = rb + t * kRec, *rg = r + dir * kGateN;
      float dgv[8];
#pragma unroll
      for (int uu = 0; uu < 2; ++uu) {
        const int u = ug + 16 * uu;
        const float e = s.hd[t * kXs + dir * kH + u] + (uu ? gh1 : gh0);
        const float ig = rg[u], fg = rg[kH + u], gg = rg[2 * kH + u], og = rg[3 * kH + u];
        const float ct = r[kRecC + dir * kH + u];
        const float cp = st > 0 ? rb[(dir == 0 ? t - 1 : t + 1) * kRec + kRecC + dir * kH + u] : 0.0f;
        const float tc = tanh_f(ct);
        float &dc = uu ? dc1 : dc0;
        const float dov = e * tc * (og * (1.0f - og));
        dc = fmaf(e * og, 1.0f - tc * tc, dc);
        const float di = dc * gg * (ig * (1.0f - ig)), dgg = dc * ig * (1.0f - gg * gg);
        const float df = dc * cp * (fg * (1.0f - fg));
        dc *= fg;
        rg[u] = di; rg[kH + u] = df; rg[2 * kH + u] = dgg; rg[3 * kH + u] = dov;
        dgv[0 + uu] = di; dgv[2 + uu] = df; dgv[4 + uu] = dgg; dgv[6 + uu] = dov;
      }
      float *dgd = s.dg + dir * kGateN;
      *reinterpret_cast<float4 *>(dgd + ug * 8) = make_float4(dgv[0], dgv[1], dgv[2], dgv[3]);
      *reinterpret_cast<float4 *>(dgd + ug * 8 + 4) = make_float4(dgv[4], dgv[5], dgv[6], dgv[7]);
      __syncwarp();
      if (st > 0) {
        // dh_{s-1} = W_hh^T dgates at units ug, ug + 16: row 64 + u of the direction's image holds the 128 gate
        // columns of h unit u; each lane starts at its own column quad, so a quarter-warp's loads hit distinct banks
        float p0 = 0.0f, p1 = 0.0f;
#pragma unroll 4
        for (int c = 0; c < kGateN / 4; ++c) {
          const int q = ((c + ug) & (kGateN / 4 - 1)) * 4;
          const float4 d = *reinterpret_cast<const float4 *>(dgd + q);
          const float4 a = *reinterpret_cast<const float4 *>(Wd + (kHid + ug) * kGateN + q);
          const float4 a2 = *reinterpret_cast<const float4 *>(Wd + (kHid + ug + 16) * kGateN + q);
          p0 = fmaf(a.x, d.x, p0); p0 = fmaf(a.y, d.y, p0); p0 = fmaf(a.z, d.z, p0); p0 = fmaf(a.w, d.w, p0);
          p1 = fmaf(a2.x, d.x, p1); p1 = fmaf(a2.y, d.y, p1); p1 = fmaf(a2.z, d.z, p1); p1 = fmaf(a2.w, d.w, p1);
        }
        gh0 = p0; gh1 = p1;
      }
      __syncwarp();  // s.dg is rewritten by the next step
    }

    // ---- per agent: dx = W_ih^T dgates over both directions, the dense1 relu, dobs = W1^T dz1
    for (int t = 0; t < N; ++t) {
      float *r = rb + t * kRec;
      for (int i = lane; i < 2 * kGateN; i += 32) {  // reference row order -> the image's column order
        const int d = i >> 7, gate = (i >> 5) & 3, unit = i & 31;
        s.dg[d * kGateN + (unit & 15) * 8 + gate * 2 + (unit >> 4)] = r[i];
      }
      __syncwarp();
      float dx0 = 0.0f, dx1 = 0.0f;
#pragma unroll
      for (int d = 0; d < 2; ++d) {
        const float *Wi = sw + w.off_wg[d], *dgd = s.dg + d * kGateN;
#pragma unroll 4
        for (int c = 0; c < kGateN / 4; ++c) {
          const int q = ((c + lane) & (kGateN / 4 - 1)) * 4;
          const float4 g = *reinterpret_cast<const float4 *>(dgd + q);
          const float4 a = *reinterpret_cast<const float4 *>(Wi + lane * kGateN + q);
          const float4 a2 = *reinterpret_cast<const float4 *>(Wi + (lane + 32) * kGateN + q);
          dx0 = fmaf(a.x, g.x, dx0); dx0 = fmaf(a.y, g.y, dx0); dx0 = fmaf(a.z, g.z, dx0); dx0 = fmaf(a.w, g.w, dx0);
          dx1 = fmaf(a2.x, g.x, dx1); dx1 = fmaf(a2.y, g.y, dx1); dx1 = fmaf(a2.z, g.z, dx1); dx1 = fmaf(a2.w, g.w, dx1);
        }
      }
      // relu(dense1): the gradient passes where x = relu(z1) > 0
      const float dz0 = s.x[t * kXs + lane] > 0.0f ? dx0 : 0.0f, dz1 = s.x[t * kXs + lane + 32] > 0.0f ? dx1 : 0.0f;
      r[kRecC + lane] = dz0; r[kRecC + lane + 32] = dz1;  // c_t is not read again
      if (dobs != nullptr) {
        s.dz[lane] = dz0; s.dz[lane + 32] = dz1;
        __syncwarp();
        // dobs_k = dense1^T dz1 at k = lane, lane + 32 (row k of the dense1 image holds its 64 units)
        for (int k = lane; k < D; k += 32) {
          float v = 0.0f;
#pragma unroll 4
          for (int c = 0; c < kHid / 4; ++c) {
            const int q = ((c + lane) & (kHid / 4 - 1)) * 4;
            const float4 z = *reinterpret_cast<const float4 *>(s.dz + q);
            const float4 wv = *reinterpret_cast<const float4 *>(W1 + k * kHid + q);
            v = fmaf(wv.x, z.x, v); v = fmaf(wv.y, z.y, v); v = fmaf(wv.z, z.z, v); v = fmaf(wv.w, z.w, v);
          }
          dobs[(b * N + t) * D + k] = v;
        }
      }
      __syncwarp();  // s.dg / s.dz are rewritten for the next agent
    }
  }
}

namespace {

// Where everything lives: the workspace is [rows][kRec] records, then [nchunk][nout] partials; the partial vector
// holds W_ih, W_hh and gate bias per direction, dense1 w / b, both heads' w / b, dense3 w / b.
struct GradPlan {
  int64_t rows, off_part, floats;
  int nchunk, nout;
  int o_wih[2], o_whh[2], o_bg[2], o_w1, o_b1, o_w2, o_b2, o_w3, o_b3;
};

GradPlan grad_plan(const ActorDev &w, int64_t B, int N) {
  GradPlan p;
  p.rows = B * N;
  p.nchunk = grad_chunks(p.rows);
  const int D3 = w.has_model ? w.D : 0;
  int off = 0;
  for (int d = 0; d < 2; ++d) {
    p.o_wih[d] = off; off += kGateN * kHid;
    p.o_whh[d] = off; off += kGateN * kH;
    p.o_bg[d] = off; off += kGateN;
  }
  p.o_w1 = off; off += kHid * w.D;
  p.o_b1 = off; off += kHid;
  p.o_w2 = off; off += w.A * kHid;
  p.o_b2 = off; off += w.A;
  p.o_w3 = off; off += D3 * kHid;
  p.o_b3 = off; off += D3;
  p.nout = (off + 63) / 64 * 64;
  p.off_part = p.rows * kRec;
  p.floats = p.off_part + (int64_t)p.nchunk * p.nout;
  return p;
}

}  // namespace

int64_t actor_backward_bytes(const ActorDev &w, int64_t B, int N) {
  return B <= 0 ? 0 : grad_plan(w, B, N).floats * (int64_t)sizeof(float);
}

cudaError_t launch_actor_backward(const ActorDev &w, const float *obs, int64_t B, int N, const float *dlogits,
                                  const float *dnext_state, float *dobs, const ActorGrads &g, void *workspace,
                                  cudaStream_t st) {
  if (B <= 0) return cudaSuccess;
  if (!actor_supported(N)) return cudaErrorInvalidValue;
  const GradPlan p = grad_plan(w, B, N);
  float *ws = static_cast<float *>(workspace);
  const int dev = current_device();
  const size_t smem = (w.smem_floats + kActorMaxA * kHid + (w.has_model ? w.D * kHid : 0)) * sizeof(float) +
                      kAgWarps * sizeof(ActorGradSmem) + 16;
  cudaError_t e = ensure_smem<k_actor_backward>(smem, dev);
  if (e != cudaSuccess) return e;
  const int nsm = sm_count(dev);
  const int64_t want = (B + kAgWarps - 1) / kAgWarps;
  k_actor_backward<<<(int)(want < nsm ? want : nsm), kAgThreads, smem, st>>>(w, obs, B, N, dlogits, dnext_state, dobs,
                                                                            ws);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;

  GradSegs segs = {};
  auto seg = [&](float *dst, int src, int n) {
    if (dst != nullptr) segs.s[segs.nseg++] = GradSeg{dst, src, n};
  };
  const int H = kHid, A0 = w.A0, A1 = w.A1, D = w.D;
  const bool d3 = dnext_state != nullptr;
  seg(g.dense1_w, p.o_w1, H * D);
  seg(g.dense1_b, p.o_b1, H);
  seg(g.w_ih, p.o_wih[0], kGateN * H);
  seg(g.w_hh, p.o_whh[0], kGateN * kH);
  seg(g.b_ih, p.o_bg[0], kGateN);
  seg(g.b_hh, p.o_bg[0], kGateN);
  seg(g.w_ih_r, p.o_wih[1], kGateN * H);
  seg(g.w_hh_r, p.o_whh[1], kGateN * kH);
  seg(g.b_ih_r, p.o_bg[1], kGateN);
  seg(g.b_hh_r, p.o_bg[1], kGateN);
  seg(g.dense2_w, p.o_w2, A0 * H);  // the heads' tile is [A0 + A1][64]: dense2 / dense2_1 rows first
  seg(g.dense2_b, p.o_b2, A0);
  seg(g.dense2b_w, p.o_w2 + A0 * H, A1 * H);
  seg(g.dense2b_b, p.o_b2 + A0, A1);
  seg(g.dense3_w, d3 ? p.o_w3 : -1, D * H);
  seg(g.dense3_b, d3 ? p.o_b3 : -1, D);
  if (segs.nseg == 0) return cudaSuccess;

  const float *rec = ws;
  GradTiles tiles = {};
  int nt = 0;
  for (int d = 0; d < 2; ++d)
    for (int mt = 0; mt < kGateN / 64; ++mt) {  // dW_ih = sum dgates^T x (+ the gate bias), dW_hh = sum dgates^T h_{s-1}
      const float *dgt = rec + d * kGateN + mt * 64;
      tiles.t[nt++] = GradTile{dgt, rec + kRecX, p.rows, kRec, kRec, 64, H, p.o_wih[d] + mt * 64 * H, H, p.o_bg[d] + mt * 64};
      tiles.t[nt++] = GradTile{dgt, rec + kRecHp + d * kH, p.rows, kRec, kRec, 64, kH, p.o_whh[d] + mt * 64 * kH, kH, -1};
    }
  tiles.t[nt++] = GradTile{rec + kRecC, obs, p.rows, kRec, D, H, D, p.o_w1, D, p.o_b1};                // dense1
  tiles.t[nt++] = GradTile{dlogits, rec + kRecH, p.rows, w.A, kRec, w.A, H, p.o_w2, H, p.o_b2};        // heads
  if (d3) tiles.t[nt++] = GradTile{dnext_state, rec + kRecH, p.rows, D, kRec, D, H, p.o_w3, H, p.o_b3};  // dense3
  tiles.nchunk = p.nchunk;
  tiles.nout = p.nout;
  return launch_grad_reduce(tiles, nt, segs, ws + p.off_part, st);
}

}  // namespace mpe
