// Host-side interface of the actor kernels (actor_kernels.cu, tc_kernels.cu; backward: actor_grad_kernels.cu) used
// by cabi.cu.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/mpe_b200.h"
#include "env_launch.h"

namespace mpe {

constexpr int kActorMaxD = 64;  // obs_dim bound (simple_spread N=12 has 28)
constexpr int kActorMaxA = 16;  // act0 + act1 bound (simple_reference has 5 + 10)
constexpr int kHid = 64;        // dense1 width / BiLSTM output width
constexpr int kH = 32;          // LSTM hidden size per direction
constexpr int kGateK = 96;      // [h1 (64) | h_prev (32)] contraction length of one LSTM step
constexpr int kGateN = 128;     // i, f, g, o gates x 32 units

// Device-resident packed weights.  Everything is stored k-major ("transposed") so that a thread's
// output columns are contiguous:  Wg[dir][k][col'] with col' = ug*8 + gate*2 + uu holding the
// reference row gate*32 + (ug + 16*uu) of [weight_ih | weight_hh]; biases b_ih + b_hh pre-summed.
// fp16 hi/lo weight image of the tensor-core path (byte offsets; see tc_kernels.cu)
// dense2 heads of one direction as a B operand [K = 32 units][24 rows]: head entry a < 8 in row 8 + a, rows 0-7 and
// 16-23 zero, so that the N = 16 operand starting at row 8 / row 0 puts the heads into columns 0-7 / 8-15
constexpr int kW2Rows = 24;
constexpr uint32_t kW2Bytes = (kH / 8) * kW2Rows * 16;
struct TcDev {
  unsigned char *blob = nullptr;
  uint32_t bytes = 0;
  int D = 0, Kx = 0, A0 = 0, A1 = 0, A = 0;
  uint32_t off_wih[2][2] = {}, off_whh[2][2] = {}, off_w1[2] = {}, off_w2[2][2] = {};
  uint32_t off_w2f = 0, off_bg = 0, off_b1 = 0, off_b2 = 0;
  float *scratch = nullptr;  // tc_scratch_floats(SMs): per-CTA dense2 shares (teams of > 3 agents, two-head actors)
};

enum { kImplAuto = 0, kImplSimt = 1, kImplTc = 2 };

struct ActorDev {
  TcDev tc;
  int impl = kImplAuto;
  float *blob = nullptr;
  size_t blob_floats = 0;
  size_t smem_floats = 0;  // leading part of the blob a CTA stages in shared memory (everything but the dense3 head)
  int D = 0, A0 = 0, A1 = 0, A = 0, Apad = 0, Dpad = 0, has_model = 0;
  int off_wg[2] = {0, 0};  // [96][128]
  int off_bg = 0;          // [2][128]
  int off_w1 = 0;          // [D][64]
  int off_b1 = 0;          // [64]
  int off_w2 = 0;          // [64][Apad]   (dense2 | dense2_1 ++ dense2_2)
  int off_b2 = 0;          // [Apad]
  int off_w3 = 0;          // [64][Dpad]   (dense3)
  int off_b3 = 0;          // [Dpad]
};

struct ActorIO {
  const float *obs = nullptr;     // [B][N][D]
  const float *gumbel = nullptr;  // [B][N][A] or null (Philox)
  float *logits = nullptr;        // [B][N][A]
  float *next_state = nullptr;    // [B][N][D]
  int32_t *act_u = nullptr, *act_c = nullptr;  // [B][N]
  float *onehot = nullptr;        // [B][N][A]
  float *hcat = nullptr;          // [B][N][64] relu(BiLSTM output): tensor-core path only, feeds launch_dense3
  int64_t B = 0, gid0 = 0;
  int32_t N = 0;
  uint64_t seed = 0, step = 0;
};

struct RolloutIO {
  int32_t T = 0;
  uint64_t step0 = 0;
  float *obs_next = nullptr;  // [T][B][N][D]
  float *rew = nullptr;       // [T][B][N]
  int32_t *act_u = nullptr, *act_c = nullptr;  // [T][B][N]
  int32_t *info_i = nullptr;  // [T][B][N+1] benchmark_data: collisions per agent, occupied landmarks (mpe_step's info_i)
  float *info_f = nullptr;    // [T][B] benchmark_data: sum of min distances (mpe_step's info_f)
};

void actor_layout(int D, int A0, int A1, bool has_model, ActorDev *out);
bool actor_supported(int N);
bool rollout_supported(int scenario, int N);
cudaError_t launch_actor_forward(const ActorDev &w, const ActorIO &io, cudaStream_t st);
// tensor-core path (tc_kernels.cu)
void tc_layout(int D, int A0, int A1, TcDev *out);
bool tc_actor_supported(const TcDev &w, int N);
bool tc_rollout_supported(const TcDev &w, int N);
size_t tc_scratch_floats(int sm_count);
cudaError_t launch_actor_forward_tc(const TcDev &w, const ActorIO &io, cudaStream_t st);
cudaError_t launch_rollout_tc(const EnvStateAny &env, const TcDev &w, const RolloutIO &io, cudaStream_t st);
// Packs the actor's images from DEVICE pointers to the reference's tensors (pack_kernels.cu): d.blob always, d.tc.blob
// when d.tc.Kx > 0.  dense2b_* are read only when A1 > 0, dense3_* only with the model head.
cudaError_t launch_actor_pack(const ActorDev &d, const ActorWeights &src, cudaStream_t st);
// next_state = dense3(hcat): the "+model" head (ac_network_model_multi_gumbel.py:49,65) on top of the tensor-core forward
cudaError_t launch_dense3(const ActorDev &w, const float *hcat, int64_t rows, float *next_state, cudaStream_t st);
// Bytes of the workspace launch_actor_backward needs for B samples of N agents (0 for B <= 0).
int64_t actor_backward_bytes(const ActorDev &w, int64_t B, int N);
// Gradients of the FFMA forward's logits / next_state: dlogits [B][N][A] upstream, dnext_state [B][N][D] (NULL: zero),
// dobs [B][N][D] and the non-NULL fields of `g` ([out][in] layout) overwritten.  `workspace` holds
// actor_backward_bytes(w, B, N) bytes of device memory.
cudaError_t launch_actor_backward(const ActorDev &w, const float *obs, int64_t B, int N, const float *dlogits,
                                  const float *dnext_state, float *dobs, const ActorGrads &g, void *workspace,
                                  cudaStream_t st);

}  // namespace mpe
