// Host-side interface of the replay kernels (replay_kernels.cu) used by cabi.cu.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace mpe {

// One transition = one contiguous record of the ring, so that a uniformly sampled transition is ONE DRAM burst:
//   [obs N*D f32][obs_next N*D f32][shared reward f32][done f32][act_u N int8][act_c N int8] padded to 16 B
// (256 B for simple_spread N = 3).  With six separate arrays a sample touched 2 x (4-5) + 4 sectors for 250 B of payload.
struct ReplayDev {
  unsigned char *ring = nullptr;  // [capacity][rec_bytes]
  int64_t capacity = 0, rec_bytes = 0;
  int32_t N = 0, D = 0, A0 = 0, A1 = 0;
  __host__ __device__ int64_t off_next() const { return (int64_t)N * D * 4; }
  __host__ __device__ int64_t off_rew() const { return (int64_t)N * D * 8; }
  __host__ __device__ int64_t off_done() const { return off_rew() + 4; }
  __host__ __device__ int64_t off_au() const { return off_rew() + 8; }
  __host__ __device__ int64_t off_ac() const { return off_au() + N; }
  __host__ __device__ static int64_t record_bytes(int N, int D) { return ((int64_t)N * D * 8 + 8 + 2 * N + 15) / 16 * 16; }
};

// add stages at least one whole record in shared memory; 48 KB is what a launch gets without opting in to more
constexpr int64_t kReplayMaxRecordBytes = 48 * 1024;

cudaError_t launch_replay_add(const ReplayDev &r, int64_t head, int64_t B, const float *obs, const int32_t *act_u,
                              const int32_t *act_c, const float *rew, const float *obs_next, const float *done,
                              cudaStream_t st);
// T steps of a rollout in one launch: step t's transitions are (t == 0 ? obs0 : obs_next[t-1], act_u[t], act_c[t],
// rew[t], obs_next[t]) with done = 0, [T][B][...] sources; transition first + t*B + b goes to slot (head + that) %
// capacity, and those before keep_from (overwritten later in the same call) are not written.
cudaError_t launch_replay_add_steps(const ReplayDev &r, int64_t head, int64_t B, int32_t T, int64_t first,
                                    int64_t keep_from, const float *obs0, const float *obs_next, const int32_t *act_u,
                                    const int32_t *act_c, const float *rew, cudaStream_t st);
cudaError_t launch_replay_make_index(int64_t size, int64_t batch, uint64_t seed, uint64_t counter, int64_t *idx,
                                     cudaStream_t st);
cudaError_t launch_replay_gather(const ReplayDev &r, int64_t size, int64_t batch, const int64_t *idx, float *obs, float *act_onehot,
                                 float *rew, float *obs_next, float *done, cudaStream_t st);

}  // namespace mpe
