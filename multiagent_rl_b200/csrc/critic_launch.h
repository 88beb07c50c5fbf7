// Host-side interface of the critic kernels (critic_kernels.cu: forward, critic_grad_kernels.cu: backward) used by
// cabi.cu.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/mpe_b200.h"

namespace mpe {

constexpr int kCriticH = 64;        // dense1 width = LSTM input = LSTM hidden (ac_network_multi_gumbel.py:86-92)
constexpr int kCriticMaxIn = 64;    // obs_dim + sum(action widths)
constexpr int kCriticMaxAgents = 16;
constexpr int kCriticMaxOut = 4;

// Packed fp32 blob in device memory (what a CTA stages into shared memory with one bulk copy)
struct CriticDev {
  float *blob = nullptr;
  size_t blob_floats = 0;
  int32_t D = 0, A = 0, Din = 0, out = 1, has_r = 0, relu_attn = 1;
  int32_t off_w1 = 0, off_b1 = 0, off_wih = 0, off_whh = 0, off_bg = 0, off_w2 = 0, off_b2 = 0, off_w3 = 0, off_b3 = 0;
};

void critic_layout(int D, int A, int out, bool has_r, bool relu_attn, CriticDev *o);
// Packs the blob from DEVICE pointers to the reference's tensors (pack_kernels.cu); dense3_* are read only when has_r.
cudaError_t launch_critic_pack(const CriticDev &d, const CriticWeights &src, cudaStream_t st);
// obs [B][N][D], action [B][N][A] (one-hot or soft), q / r [B][out]
cudaError_t launch_critic_forward(const CriticDev &w, const float *obs, const float *action, int64_t B, int N, float *q,
                                  float *r, cudaStream_t st);
// Bytes of the workspace launch_critic_backward needs for B samples of N agents (0 for B <= 0).
int64_t critic_backward_bytes(const CriticDev &w, int64_t B, int N);
// Gradients of launch_critic_forward's function: dq / dr [B][out] upstream (dr may be NULL), dobs [B][N][D],
// daction [B][N][A] and the non-NULL fields of `g` ([out][in] layout) overwritten.  `workspace` holds
// critic_backward_bytes(w, B, N) bytes of device memory.
cudaError_t launch_critic_backward(const CriticDev &w, const float *obs, const float *action, int64_t B, int N,
                                   const float *dq, const float *dr, float *dobs, float *daction,
                                   const CriticGrads &g, void *workspace, cudaStream_t st);

}  // namespace mpe
