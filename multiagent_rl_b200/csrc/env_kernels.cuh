// Env kernels (reset / step / observe / state transposes), templated on the real type.  Included
// by env_kernels_f32.cu and env_kernels_f64.cu (the latter built with -fmad=false).
//
// Mapping: one thread per env, 128 threads per CTA.  State loads/stores are 16 B (agents) and 8 B
// (landmarks) per lane and perfectly coalesced across the warp because state is SoA over envs.
// Outputs use the caller-facing [B][N][D] layout; a warp's 32 envs form one contiguous span of it,
// so each warp stages its rows in shared memory and one lane hands the span to the TMA engine
// (cp.async.bulk shared->global): the step kernel issues no per-element global stores for obs/rew.
#pragma once
#include "env_core.cuh"
#include "env_launch.h"
#include "launch.h"

namespace mpe {
constexpr int kStepThreads = 128;
}

namespace mpe {

constexpr int kStageMaxBytes = 16384;  // per-warp obs staging above this falls back to per-agent staging
// rewards leave through a coalesced copy of the staged values instead of a second bulk store per warp (measured:
// simple_reference 0.857 -> 0.877 of HBM, the others unchanged)
constexpr bool kStageRewards = false;

template <typename T, int SC, int N>
struct StageLayout {
  using Dm = Dims<SC, N>;
  static constexpr bool kFull = (32 * Dm::R * (int)sizeof(T) <= kStageMaxBytes);
  static constexpr int kObsElems = kFull ? 32 * Dm::R : 32 * Dm::D;
  static constexpr int kRewElems = 32 * N;
  static constexpr int kWarpBytes = (kObsElems + kRewElems) * (int)sizeof(T);  // multiple of 128
  static constexpr int kBlockBytes = kWarpBytes * (kStepThreads / 32);
};

// Write one warp's obs rows + rewards.  `full` (warp-uniform): all 32 lanes own a valid env.
template <typename T, int SC, int N>
__device__ __forceinline__ void emit_outputs(const Env<T, SC, N> &e, const T (*comm)[10], const T *r,
                                             bool want_rew, T *obs, T *rew, int64_t b0, int lane, bool full,
                                             bool active, unsigned char *smem_warp) {
  using Dm = Dims<SC, N>;
  using SL = StageLayout<T, SC, N>;
  constexpr int D = Dm::D, R = Dm::R;
  T *st_obs = reinterpret_cast<T *>(smem_warp);
  T *st_rew = st_obs + SL::kObsElems;
  // TMA bulk stores need 16 B aligned global addresses (warp spans are multiples of 128 B)
  const bool obs_tma = SL::kFull && (reinterpret_cast<uintptr_t>(obs) & 15) == 0;
  const bool rew_tma = kStageRewards && (reinterpret_cast<uintptr_t>(rew) & 15) == 0;
  if (full) {
    bool issued = false;
    if (obs != nullptr) {
      if (SL::kFull) {
#pragma unroll
        for (int i = 0; i < N; ++i) e.obs_row(i, st_obs + lane * R + i * D, SC == kReference ? comm[1 - (i & 1)] : nullptr);
      }
    }
    if (want_rew) {
#pragma unroll
      for (int i = 0; i < N; ++i) st_rew[lane * N + i] = r[i];
    }
    if ((obs != nullptr && SL::kFull) || want_rew) {
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        if (obs != nullptr && obs_tma) bulk_store(obs + b0 * R, st_obs, 32 * R * sizeof(T));
        if (want_rew && rew_tma) bulk_store(rew + b0 * N, st_rew, 32 * N * sizeof(T));
        bulk_commit();
        issued = true;
      }
      if (obs != nullptr && SL::kFull && !obs_tma)
        for (int i = lane; i < 32 * R; i += 32) obs[b0 * R + i] = st_obs[i];
      if (want_rew && !rew_tma)
        for (int i = lane; i < 32 * N; i += 32) rew[b0 * N + i] = st_rew[i];
    }
    if (obs != nullptr && !SL::kFull) {
      // large N: stage one agent at a time, copy rows out with coalesced-per-row scalar stores
#pragma unroll 1
      for (int i = 0; i < N; ++i) {
        __syncwarp();
        // obs_row needs a compile-time agent index for register arrays: select by unrolled compare
#pragma unroll
        for (int ii = 0; ii < N; ++ii)
          if (ii == i) e.obs_row(ii, st_obs + lane * D, nullptr);
        __syncwarp();
        for (int idx = lane; idx < 32 * D; idx += 32) {
          const int env = idx / D, j = idx - env * D;
          obs[(b0 + env) * R + i * D + j] = st_obs[idx];
        }
      }
    }
    if (issued) bulk_wait_read_all();
  } else if (active) {
    const int64_t b = b0 + lane;
    if (obs != nullptr) {
#pragma unroll
      for (int i = 0; i < N; ++i) e.obs_row(i, obs + b * R + i * D, SC == kReference ? comm[1 - (i & 1)] : nullptr);
    }
    if (want_rew) {
#pragma unroll
      for (int i = 0; i < N; ++i) rew[b * N + i] = r[i];
    }
  }
}

template <typename T, int SC, int N>
__device__ __forceinline__ void load_comm(const EnvState<T> &s, int64_t b, T (*comm)[10]) {
  if (SC == kReference) {
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int k = 0; k < 10; ++k) comm[i][k] = s.comm[((int64_t)i * 10 + k) * s.B + b];
  }
}
template <typename T, int SC, int N>
__device__ __forceinline__ void store_comm(const EnvState<T> &s, int64_t b, const T (*comm)[10]) {
  if (SC == kReference) {
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int k = 0; k < 10; ++k) s.comm[((int64_t)i * 10 + k) * s.B + b] = comm[i][k];
  }
}

// ---------------------------------------------------------------------------------------------
// env.reset(): Scenario.reset_world for the masked envs, then (optionally) the observation.
// ---------------------------------------------------------------------------------------------
template <typename T, int SC, int N>
__global__ void __launch_bounds__(kStepThreads) k_reset(EnvState<T> s, const uint8_t *mask, T *obs, int auto_len) {
  extern __shared__ __align__(128) unsigned char smem[];
  using SL = StageLayout<T, SC, N>;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t b0 = (int64_t)blockIdx.x * kStepThreads + warp * 32;
  const int64_t b = b0 + lane;
  const bool active = b < s.B;
  const bool full = b0 + 32 <= s.B;
  Env<T, SC, N> e;
  T comm[2][10];
  double ret = 0.0, n_ep = 0.0, n_steps = 0.0;
  if (active) {
    // auto_len > 0: only envs whose episode has reached auto_len steps (experiments/run.py:50,59-60)
    const bool doit = (mask == nullptr || mask[b] != 0) && (auto_len <= 0 || s.tstep[b] >= auto_len);
    if (doit) {
      const uint32_t ep = s.episode[b] + 1u;
      s.episode[b] = ep;
      e.reset(s.seed, (uint64_t)(s.gid0 + b), ep);
      e.store_agents(s, b);
      e.store_world(s, b);
      if (SC == kReference) {
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
          for (int k = 0; k < 10; ++k) comm[i][k] = (T)0;
        store_comm<T, SC, N>(s, b, comm);
      }
      const int t = s.tstep[b];
      if (s.track && t > 0) { ret = (double)s.ep_ret[b]; n_ep = 1.0; n_steps = (double)t; }
      s.tstep[b] = 0;
      s.ep_ret[b] = (T)0;
    } else if (obs != nullptr) {
      e.load(s, b);
      load_comm<T, SC, N>(s, b, comm);
    }
  }
  if (s.track) fold_stats(s.stats, ret, n_ep, n_steps);
  if (obs != nullptr)
    emit_outputs<T, SC, N>(e, comm, nullptr, false, obs, nullptr, b0, lane, full, active, smem + warp * SL::kWarpBytes);
}

template <typename T, int SC, int N>
__global__ void __launch_bounds__(kStepThreads) k_observe(EnvState<T> s, T *obs) {
  extern __shared__ __align__(128) unsigned char smem[];
  using SL = StageLayout<T, SC, N>;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t b0 = (int64_t)blockIdx.x * kStepThreads + warp * 32;
  const int64_t b = b0 + lane;
  const bool active = b < s.B;
  const bool full = b0 + 32 <= s.B;
  Env<T, SC, N> e;
  T comm[2][10];
  if (active) {
    e.load(s, b);
    load_comm<T, SC, N>(s, b, comm);
  }
  emit_outputs<T, SC, N>(e, comm, nullptr, false, obs, nullptr, b0, lane, full, active, smem + warp * SL::kWarpBytes);
}

// ---------------------------------------------------------------------------------------------
// env.step(action_n): _set_action -> World.step -> observation + reward for every agent.
// ---------------------------------------------------------------------------------------------
template <typename T, int SC, int N>
__global__ void __launch_bounds__(kStepThreads)
    k_step(EnvState<T> s, const int32_t *__restrict__ act_u, const int32_t *__restrict__ act_c,
           const T *__restrict__ comm_vec, T *__restrict__ obs, T *__restrict__ rew, uint8_t *__restrict__ done,
           int32_t *__restrict__ info_i, T *__restrict__ info_f) {
  extern __shared__ __align__(128) unsigned char smem[];
  using SL = StageLayout<T, SC, N>;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t b0 = (int64_t)blockIdx.x * kStepThreads + warp * 32;
  const int64_t b = b0 + lane;
  const bool active = b < s.B;
  const bool full = b0 + 32 <= s.B;
  Env<T, SC, N> e;
  T comm[2][10];
  T r[N];
  if (active) {
    e.load(s, b);
    int au[N];
#pragma unroll
    for (int i = 0; i < N; ++i) au[i] = act_u[b * N + i];
    e.physics(au, s);
    e.store_agents(s, b);
    if (SC == kReference) {  // World.update_agent_state: state.c = action.c
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const int ci = (comm_vec == nullptr && act_c != nullptr) ? act_c[b * N + i] : -1;
#pragma unroll
        for (int k = 0; k < 10; ++k)
          comm[i][k] = comm_vec != nullptr ? comm_vec[(b * N + i) * 10 + k] : (k == ci ? (T)1 : (T)0);
      }
      store_comm<T, SC, N>(s, b, comm);
    }
    int coll[N], occ;
    T md;
    e.reward(r, coll, occ, md, s);
    if (s.track) {
      T sum = (T)0;
#pragma unroll
      for (int i = 0; i < N; ++i) sum += r[i];
      s.ep_ret[b] += sum;
      s.tstep[b] += 1;
    }
    if (info_i != nullptr) {
#pragma unroll
      for (int i = 0; i < N; ++i) info_i[b * (N + 1) + i] = coll[i];
      info_i[b * (N + 1) + N] = occ;
    }
    if (info_f != nullptr) info_f[b] = md;
  }
  if (done != nullptr) {  // no done_callback (experiments/scenarios.py:186-190): always False
    // a full warp's span is 32*N bytes at done + b0*N, and b0*N is a multiple of 32: when `done` itself is
    // 4 B aligned the span can be zeroed with 32-bit stores.  A caller's `done` may sit at any byte offset
    // (a slice of a [T][B][N] record at odd B*N), so otherwise every env stores its own bytes.
    if (full && (reinterpret_cast<uintptr_t>(done) & 3) == 0) {
      uint32_t *d32 = reinterpret_cast<uint32_t *>(done + b0 * N);
      for (int k = lane; k < 8 * N; k += 32) d32[k] = 0u;
    } else if (active) {
#pragma unroll
      for (int i = 0; i < N; ++i) done[b * N + i] = 0;
    }
  }
  emit_outputs<T, SC, N>(e, comm, r, rew != nullptr, obs, rew, b0, lane, full, active, smem + warp * SL::kWarpBytes);
}

}  // namespace mpe
#include "env_group.cuh"
#include "env_treasure.cuh"
namespace mpe {

// ---------------------------------------------------------------------------------------------
// state injection / readback: caller layout [B][N][2] <-> device SoA.  Runtime N (not hot).
// ---------------------------------------------------------------------------------------------
template <typename T>
__global__ void k_set_state(EnvState<T> s, int N, int L, int dimc, const T *pos, const T *vel, const T *lm,
                            const int32_t *goal, int raw_goal) {
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= s.B) return;
  for (int i = 0; i < N; ++i) {
    T *p = s.pv + ((int64_t)i * s.B + b) * 4;
    if (pos != nullptr) { p[0] = pos[(b * N + i) * 2]; p[1] = pos[(b * N + i) * 2 + 1]; }
    if (vel != nullptr) { p[2] = vel[(b * N + i) * 2]; p[3] = vel[(b * N + i) * 2 + 1]; }
  }
  if (lm != nullptr)
    for (int l = 0; l < L; ++l) {
      s.lm[((int64_t)l * s.B + b) * 2] = lm[(b * L + l) * 2];
      s.lm[((int64_t)l * s.B + b) * 2 + 1] = lm[(b * L + l) * 2 + 1];
    }
  if (goal != nullptr && s.goal != nullptr) {
    const int g0 = goal[b * N], g1 = N > 1 ? goal[b * N + 1] : -1;
    s.goal[b] = raw_goal ? g0 : ((g0 & 0xFF) | ((g1 & 0xFF) << 8));  // raw: the treasure scenario's state word
  }
  if (s.comm != nullptr)
    for (int k = 0; k < N * dimc; ++k) s.comm[(int64_t)k * s.B + b] = (T)0;
}

template <typename T>
__global__ void k_get_state(EnvState<T> s, int N, int L, T *pos, T *vel, T *lm, int32_t *goal, int raw_goal) {
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= s.B) return;
  for (int i = 0; i < N; ++i) {
    const T *p = s.pv + ((int64_t)i * s.B + b) * 4;
    if (pos != nullptr) { pos[(b * N + i) * 2] = p[0]; pos[(b * N + i) * 2 + 1] = p[1]; }
    if (vel != nullptr) { vel[(b * N + i) * 2] = p[2]; vel[(b * N + i) * 2 + 1] = p[3]; }
  }
  if (lm != nullptr)
    for (int l = 0; l < L; ++l) {
      lm[(b * L + l) * 2] = s.lm[((int64_t)l * s.B + b) * 2];
      lm[(b * L + l) * 2 + 1] = s.lm[((int64_t)l * s.B + b) * 2 + 1];
    }
  if (goal != nullptr) {
    for (int i = 0; i < N; ++i) goal[b * N + i] = -1;
    if (s.goal != nullptr && raw_goal) {
      goal[b * N] = s.goal[b];
    } else if (s.goal != nullptr) {
      const int32_t g = s.goal[b];
      const int g0 = g & 0xFF, g1 = (g >> 8) & 0xFF;
      goal[b * N] = g0 == 0xFF ? -1 : g0;
      if (N > 1) goal[b * N + 1] = g1 == 0xFF ? -1 : g1;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// host-side dispatch over (scenario, N)
// ---------------------------------------------------------------------------------------------
#define MPE_DISPATCH(a, CALL)                                                       \
  do {                                                                              \
    if ((a).scenario == kSpread) {                                                  \
      switch ((a).N) {                                                              \
        case 1: CALL(kSpread, 1); break;                                            \
        case 2: CALL(kSpread, 2); break;                                            \
        case 3: CALL(kSpread, 3); break;                                            \
        case 4: CALL(kSpread, 4); break;                                            \
        case 5: CALL(kSpread, 5); break;                                            \
        default: return cudaErrorInvalidValue;                                      \
      }                                                                             \
    } else if ((a).scenario == kReference) {                                        \
      CALL(kReference, 2);                                                          \
    } else if ((a).scenario == kSpeaker) {                                          \
      CALL(kSpeaker, 2);                                                            \
    } else {                                                                        \
      return cudaErrorInvalidValue;                                                 \
    }                                                                               \
  } while (0)

// G-lanes-per-env families: GRP(N, G) for every team size of 6..12
#define MPE_DISPATCH_GRP(a, GRP) \
  do {                           \
    switch ((a).N) {             \
      case 6: GRP(6, 2)          \
      case 7: GRP(7, 7)          \
      case 8: GRP(8, 4)          \
      case 9: GRP(9, 3)          \
      case 10: GRP(10, 5)        \
      case 11: GRP(11, 11)       \
      case 12: GRP(12, 4)        \
      default: return cudaErrorInvalidValue; \
    }                            \
  } while (0)

#define MPE_GRP_RESET(NN, GG, DO_RESET)                                                                            \
  {                                                                                                                \
    using GL = GroupLayout<T, NN, GG>;                                                                             \
    constexpr int sm = GL::kBlockBytes;                                                                            \
    cudaError_t err = ensure_smem<k_reset_grp<T, NN, GG>>(sm);                                                       \
    if (err != cudaSuccess) return err;                                                                            \
    const int64_t per_block = (int64_t)GL::EPW * (kStepThreads / 32);                                              \
    k_reset_grp<T, NN, GG><<<(unsigned)((a.B + per_block - 1) / per_block), kStepThreads, sm, st>>>(               \
        typed<T>(a), mask, static_cast<T *>(obs), auto_len, DO_RESET);                                             \
    return cudaGetLastError();                                                                                     \
  }

// fullobs_collect_treasure: one kernel template, MODE = step / reset / observe (env_treasure.cuh)
template <typename T, int MODE>
cudaError_t launch_treasure_t(const EnvStateAny &a, const int32_t *act_u, const uint8_t *mask, int auto_len, void *obs,
                              void *rew, uint8_t *done, int32_t *info_i, cudaStream_t st) {
  constexpr int sm = TrLayout<T>::kBlockBytes;
  cudaError_t err = ensure_smem<k_treasure<T, MODE>>(sm);
  if (err != cudaSuccess) return err;
  const int64_t per_block = TrLayout<T>::kEnvsPerBlock;  // 8 lanes per env
  const unsigned grid = (unsigned)((a.B + per_block - 1) / per_block);
  k_treasure<T, MODE><<<grid, kStepThreads, sm, st>>>(typed<T>(a), act_u, mask, auto_len, static_cast<T *>(obs),
                                                      static_cast<T *>(rew), done, info_i);
  return cudaGetLastError();
}

template <typename T>
cudaError_t launch_reset_t(const EnvStateAny &a, const uint8_t *mask, void *obs, int auto_len, cudaStream_t st) {
  if (a.B <= 0) return cudaSuccess;
  if (a.scenario == kTreasure) return launch_treasure_t<T, 1>(a, nullptr, mask, auto_len, obs, nullptr, nullptr, nullptr, st);
  if (a.scenario == kSpread && group_lanes(a.N) > 0) {  // G lanes per env (env_group.cuh)
#define GRP(NN, GG) MPE_GRP_RESET(NN, GG, 1)
    MPE_DISPATCH_GRP(a, GRP);
#undef GRP
  }
  const unsigned grid = (unsigned)((a.B + kStepThreads - 1) / kStepThreads);
#define CALL(SC, NN)                                                                          \
  {                                                                                           \
    constexpr int sm = StageLayout<T, SC, NN>::kBlockBytes;                                   \
    cudaError_t err = ensure_smem<k_reset<T, SC, NN>>(sm);                                      \
    if (err != cudaSuccess) return err;                                                       \
    k_reset<T, SC, NN><<<grid, kStepThreads, sm, st>>>(typed<T>(a), mask, static_cast<T *>(obs), auto_len); \
  }
  MPE_DISPATCH(a, CALL);
#undef CALL
  return cudaGetLastError();
}

template <typename T>
cudaError_t launch_observe_t(const EnvStateAny &a, void *obs, cudaStream_t st) {
  if (a.B <= 0) return cudaSuccess;
  if (a.scenario == kTreasure) return launch_treasure_t<T, 2>(a, nullptr, nullptr, 0, obs, nullptr, nullptr, nullptr, st);
  if (a.scenario == kSpread && group_lanes(a.N) > 0) {
    const uint8_t *mask = nullptr;
    const int auto_len = 0;
#define GRP(NN, GG) MPE_GRP_RESET(NN, GG, 0)
    MPE_DISPATCH_GRP(a, GRP);
#undef GRP
  }
  const unsigned grid = (unsigned)((a.B + kStepThreads - 1) / kStepThreads);
#define CALL(SC, NN)                                                                    \
  {                                                                                     \
    constexpr int sm = StageLayout<T, SC, NN>::kBlockBytes;                             \
    cudaError_t err = ensure_smem<k_observe<T, SC, NN>>(sm);                              \
    if (err != cudaSuccess) return err;                                                 \
    k_observe<T, SC, NN><<<grid, kStepThreads, sm, st>>>(typed<T>(a), static_cast<T *>(obs)); \
  }
  MPE_DISPATCH(a, CALL);
#undef CALL
  return cudaGetLastError();
}

template <typename T>
cudaError_t launch_step_t(const EnvStateAny &a, const int32_t *act_u, const int32_t *act_c, const void *comm_vec,
                          void *obs, void *rew, uint8_t *done, int32_t *info_i, void *info_f, cudaStream_t st) {
  if (a.B <= 0) return cudaSuccess;
  if (a.scenario == kTreasure) return launch_treasure_t<T, 0>(a, act_u, nullptr, 0, obs, rew, done, info_i, st);
  if (a.scenario == kSpread && group_lanes(a.N) > 0) {  // G lanes per env (env_group.cuh)
#define GRP(NN, GG)                                                                                                \
  {                                                                                                                \
    using GL = GroupLayout<T, NN, GG>;                                                                             \
    constexpr int sm = GL::kBlockBytes;                                                                            \
    cudaError_t err = ensure_smem<k_step_grp<T, NN, GG>>(sm);                                                        \
    if (err != cudaSuccess) return err;                                                                            \
    const int64_t per_block = (int64_t)GL::EPW * (kStepThreads / 32);                                              \
    k_step_grp<T, NN, GG><<<(unsigned)((a.B + per_block - 1) / per_block), kStepThreads, sm, st>>>(                \
        typed<T>(a), act_u, static_cast<T *>(obs), static_cast<T *>(rew), done, info_i, static_cast<T *>(info_f)); \
    return cudaGetLastError();                                                                                     \
  }
    MPE_DISPATCH_GRP(a, GRP);
#undef GRP
  }
  const unsigned grid = (unsigned)((a.B + kStepThreads - 1) / kStepThreads);
#define CALL(SC, NN)                                                                                         \
  {                                                                                                          \
    constexpr int sm = StageLayout<T, SC, NN>::kBlockBytes;                                                  \
    cudaError_t err = ensure_smem<k_step<T, SC, NN>>(sm);                                                      \
    if (err != cudaSuccess) return err;                                                                      \
    k_step<T, SC, NN><<<grid, kStepThreads, sm, st>>>(typed<T>(a), act_u, act_c, static_cast<const T *>(comm_vec), \
                                                      static_cast<T *>(obs), static_cast<T *>(rew), done, info_i, \
                                                      static_cast<T *>(info_f));                             \
  }
  MPE_DISPATCH(a, CALL);
#undef CALL
  return cudaGetLastError();
}

template <typename T>
cudaError_t launch_set_state_t(const EnvStateAny &a, const void *pos, const void *vel, const void *lm,
                               const int32_t *goal, cudaStream_t st) {
  if (a.B <= 0) return cudaSuccess;
  const unsigned grid = (unsigned)((a.B + 255) / 256);
  k_set_state<T><<<grid, 256, 0, st>>>(typed<T>(a), a.N, a.L, a.dimc, static_cast<const T *>(pos),
                                       static_cast<const T *>(vel), static_cast<const T *>(lm), goal,
                                       a.scenario == kTreasure ? 1 : 0);
  return cudaGetLastError();
}

template <typename T>
cudaError_t launch_get_state_t(const EnvStateAny &a, void *pos, void *vel, void *lm, int32_t *goal, cudaStream_t st) {
  if (a.B <= 0) return cudaSuccess;
  const unsigned grid = (unsigned)((a.B + 255) / 256);
  k_get_state<T><<<grid, 256, 0, st>>>(typed<T>(a), a.N, a.L, static_cast<T *>(pos), static_cast<T *>(vel),
                                       static_cast<T *>(lm), goal, a.scenario == kTreasure ? 1 : 0);
  return cudaGetLastError();
}

}  // namespace mpe
