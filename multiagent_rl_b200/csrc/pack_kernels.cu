// Weight packing on the device: the reference's row-major [out][in] fp32 tensors -> the images the forward kernels
// stage into shared memory - the actor's fp32 FFMA blob (actor_layout), its fp16 hi/lo tensor-core image (tc_layout)
// and the critic's fp32 blob (critic_layout).  This file is the only place that knows which source element lands in
// which word of an image.
//
// Gather form: one thread per 32-bit word of an image computes that word from the layout, zero padding included, so
// every word is written exactly once, nothing depends on the image's previous contents or on the order of writes, and
// nothing outside the image is written.  Sources are read with scalar loads: views into a flat parameter buffer may be
// only 4 B aligned.  The rounding is spelled out with intrinsics so that the compiler cannot contract it and the images
// do not depend on the build.  About 100 - 210 KB per load: the kernels are launch-bound.
#include <cuda_fp16.h>

#include "actor_launch.h"
#include "critic_launch.h"
#include "tc_common.cuh"

namespace mpe {

constexpr int kPackThreads = 256;

// ------------------------------------------------------------------------------------------------
// actor
// ------------------------------------------------------------------------------------------------
// dense2 heads: logit a < A0 from dense2 (dense2_1), the rest from dense2_2
__device__ __forceinline__ float head_w(const ActorWeights &w, int A0, int a, int k) {
  return a < A0 ? w.dense2_w[a * kHid + k] : w.dense2b_w[(a - A0) * kHid + k];
}
__device__ __forceinline__ float head_b(const ActorWeights &w, int A0, int a) {
  return a < A0 ? w.dense2_b[a] : w.dense2b_b[a - A0];
}
__device__ __forceinline__ float gate_bias(const ActorWeights &w, int dir, int row) {
  return __fadd_rn((dir ? w.b_ih_r : w.b_ih)[row], (dir ? w.b_hh_r : w.b_hh)[row]);
}

// Word i of the FFMA blob.  Gate column col = ug * 8 + gate * 2 + uu holds the reference row gate * 32 + ug + 16 * uu.
__device__ float actor_blob_word(const ActorDev &d, const ActorWeights &w, int i) {
  if (i < d.off_bg) {  // [dir][k][col], k < 64 from weight_ih, else weight_hh
    const int dir = i >= d.off_wg[1] ? 1 : 0, r = i - d.off_wg[dir], k = r / kGateN, col = r % kGateN;
    const int row = ((col >> 1) & 3) * kH + (col >> 3) + 16 * (col & 1);
    return k < kHid ? (dir ? w.w_ih_r : w.w_ih)[row * kHid + k] : (dir ? w.w_hh_r : w.w_hh)[row * kH + k - kHid];
  }
  if (i < d.off_w1) {  // [dir][col]: b_ih + b_hh
    const int r = i - d.off_bg, dir = r / kGateN, col = r % kGateN;
    return gate_bias(w, dir, ((col >> 1) & 3) * kH + (col >> 3) + 16 * (col & 1));
  }
  if (i < d.off_b1) {  // dense1 [k][j]
    const int r = i - d.off_w1;
    return r < d.D * kHid ? w.dense1_w[(r % kHid) * d.D + r / kHid] : 0.0f;
  }
  if (i < d.off_w2) return w.dense1_b[i - d.off_b1];
  if (i < d.off_b2) {  // dense2 heads [k][Apad]
    const int r = i - d.off_w2, a = r % d.Apad;
    return a < d.A ? head_w(w, d.A0, a, r / d.Apad) : 0.0f;
  }
  if (i < d.off_b2 + d.Apad) {
    const int a = i - d.off_b2;
    return a < d.A ? head_b(w, d.A0, a) : 0.0f;
  }
  if (!d.has_model || i < d.off_w3) return 0.0f;  // padding of the staged part
  if (i < d.off_b3) {  // dense3 [k][Dpad]
    const int r = i - d.off_w3, j = r % d.Dpad;
    return j < d.D ? w.dense3_w[j * kHid + r / d.Dpad] : 0.0f;
  }
  const int j = i - d.off_b3;
  return j < d.D ? w.dense3_b[j] : 0.0f;  // j >= Dpad: padding to the blob's end
}

// x = 16 v = hi + lo: the hi (which = 0) or lo (which = 1) half, as tc_kernels.cu's operands expect
__device__ __forceinline__ uint16_t split_part(float v, int which) {
  const float x = __fmul_rn(v, kWScale);
  const __half hi = __float2half_rn(x);
  return __half_as_ushort(which ? __float2half_rn(__fsub_rn(x, __half2float(hi))) : hi);
}

// The 32-bit word at byte o of the tensor-core image (t.Kx > 0).
__device__ uint32_t actor_tc_word(const TcDev &t, const ActorWeights &w, uint32_t o) {
  if (o < t.off_w2f) {
    // fp16 operands [K/8][rows][8]: the word holds elements k and k + 1 of one row n, k even
    uint32_t base;
    int rows, which, kind, dir = 0;
    if (o < t.off_whh[0][0]) {
      const uint32_t q = (o - t.off_wih[0][0]) / (kHid * kGateN * 2);
      dir = q >> 1; which = q & 1; base = t.off_wih[dir][which]; rows = kGateN; kind = 0;
    } else if (o < t.off_w1[0]) {
      const uint32_t q = (o - t.off_whh[0][0]) / (kH * kGateN * 2);
      dir = q >> 1; which = q & 1; base = t.off_whh[dir][which]; rows = kGateN; kind = 1;
    } else if (o < t.off_w2[0][0]) {
      which = o >= t.off_w1[1] ? 1 : 0; base = t.off_w1[which]; rows = kHid; kind = 2;
    } else {
      const uint32_t q = (o - t.off_w2[0][0]) / kW2Bytes;
      dir = q >> 1; which = q & 1; base = t.off_w2[dir][which]; rows = kW2Rows; kind = 3;
    }
    const int h = (int)(o - base) / 2, n = (h / 8) % rows, k = (h / (8 * rows)) * 8 + h % 8;
    float v0, v1;
    if (kind == 2) {  // dense1: row j = n, columns past D are zero
      v0 = k < t.D ? w.dense1_w[n * t.D + k] : 0.0f;
      v1 = k + 1 < t.D ? w.dense1_w[n * t.D + k + 1] : 0.0f;
    } else if (kind == 3) {  // dense2 heads: row n = 8 + a holds head entry a < min(A, 8), unit k of direction dir
      const int a = n - 8;
      const bool on = a >= 0 && a < 8 && a < t.A;
      v0 = on ? head_w(w, t.A0, a, dir * kH + k) : 0.0f;
      v1 = on ? head_w(w, t.A0, a, dir * kH + k + 1) : 0.0f;
    } else {  // gate column n = (u >> 1) * 8 + g * 2 + (u & 1) holds the reference row g * 32 + u
      const int row = ((n >> 1) & 3) * kH + ((n >> 3) << 1) + (n & 1);
      const float *src = kind == 0 ? (dir ? w.w_ih_r : w.w_ih) + row * kHid : (dir ? w.w_hh_r : w.w_hh) + row * kH;
      v0 = src[k]; v1 = src[k + 1];
    }
    return (uint32_t)split_part(v0, which) | ((uint32_t)split_part(v1, which) << 16);
  }
  float v = 0.0f;
  if (o < t.off_bg) {  // dense2 heads fp32 [k][16] (the FFMA heads of large teams and two-head actors)
    const int r = (int)(o - t.off_w2f) / 4, a = r % 16;
    v = a < t.A ? head_w(w, t.A0, a, r / 16) : 0.0f;
  } else if (o < t.off_b1) {  // gate biases in the ex2 argument form: (b_ih + b_hh) * (-2 | -1) * log2(e)
    const int r = (int)(o - t.off_bg) / 4, dir = r / kGateN, n = r % kGateN, g = (n >> 1) & 3;
    v = __fmul_rn(__fmul_rn(gate_bias(w, dir, g * kH + ((n >> 3) << 1) + (n & 1)), g == 2 ? -2.0f : -1.0f), kLog2e);
  } else if (o < t.off_b2) {
    v = w.dense1_b[(o - t.off_b1) / 4];
  } else if (o < t.off_b2 + 16 * 4) {
    const int a = (int)(o - t.off_b2) / 4;
    v = a < t.A ? head_b(w, t.A0, a) : 0.0f;
  }
  return __float_as_uint(v);
}

__global__ void __launch_bounds__(kPackThreads) k_actor_pack(ActorDev d, ActorWeights w) {
  const int64_t n_blob = (int64_t)d.blob_floats, n_tc = d.tc.Kx > 0 ? d.tc.bytes / 4 : 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_blob + n_tc; i += (int64_t)gridDim.x * blockDim.x) {
    if (i < n_blob) d.blob[i] = actor_blob_word(d, w, (int)i);
    else reinterpret_cast<uint32_t *>(d.tc.blob)[i - n_blob] = actor_tc_word(d.tc, w, 4 * (uint32_t)(i - n_blob));
  }
}

cudaError_t launch_actor_pack(const ActorDev &d, const ActorWeights &w, cudaStream_t st) {
  const int64_t words = (int64_t)d.blob_floats + (d.tc.Kx > 0 ? d.tc.bytes / 4 : 0);
  k_actor_pack<<<(unsigned)((words + kPackThreads - 1) / kPackThreads), kPackThreads, 0, st>>>(d, w);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// critic
// ------------------------------------------------------------------------------------------------
// Word i of the critic blob.  Gate column col = lane * 8 + gate * 2 + hi holds the reference row gate * 64 + lane + 32 hi.
__device__ float critic_blob_word(const CriticDev &d, const CriticWeights &w, int i) {
  constexpr int kG = 4 * kCriticH;
  if (i < d.off_bg) {  // weight_ih then weight_hh, each [k][col]
    const int m = i >= d.off_whh ? 1 : 0, r = i - (m ? d.off_whh : d.off_wih), col = r % kG;
    const int row = ((col >> 1) & 3) * kCriticH + (col >> 3) + 32 * (col & 1);
    return (m ? w.w_hh : w.w_ih)[row * kCriticH + r / kG];
  }
  if (i < d.off_w1) {
    const int col = i - d.off_bg, row = ((col >> 1) & 3) * kCriticH + (col >> 3) + 32 * (col & 1);
    return __fadd_rn(w.b_ih[row], w.b_hh[row]);
  }
  if (i < d.off_b1) {  // dense1 [k][j]
    const int r = i - d.off_w1;
    return r < d.Din * kCriticH ? w.dense1_w[(r % kCriticH) * d.Din + r / kCriticH] : 0.0f;
  }
  if (i < d.off_w2) return w.dense1_b[i - d.off_b1];
  if (i < d.off_b2) {  // dense2 [k][kCriticMaxOut]
    const int r = i - d.off_w2, o = r % kCriticMaxOut;
    return o < d.out ? w.dense2_w[o * kCriticH + r / kCriticMaxOut] : 0.0f;
  }
  if (i < d.off_w3) {
    const int o = i - d.off_b2;
    return o < d.out ? w.dense2_b[o] : 0.0f;
  }
  if (i < d.off_b3) {  // dense3 [k][kCriticMaxOut], "+model" critics only
    const int r = i - d.off_w3, o = r % kCriticMaxOut;
    return d.has_r && o < d.out ? w.dense3_w[o * kCriticH + r / kCriticMaxOut] : 0.0f;
  }
  const int o = i - d.off_b3;
  return d.has_r && o < d.out ? w.dense3_b[o] : 0.0f;  // o >= kCriticMaxOut: padding to the blob's end
}

__global__ void __launch_bounds__(kPackThreads) k_critic_pack(CriticDev d, CriticWeights w) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (int64_t)d.blob_floats;
       i += (int64_t)gridDim.x * blockDim.x)
    d.blob[i] = critic_blob_word(d, w, (int)i);
}

cudaError_t launch_critic_pack(const CriticDev &d, const CriticWeights &w, cudaStream_t st) {
  k_critic_pack<<<(unsigned)((d.blob_floats + kPackThreads - 1) / kPackThreads), kPackThreads, 0, st>>>(d, w);
  return cudaGetLastError();
}

}  // namespace mpe
