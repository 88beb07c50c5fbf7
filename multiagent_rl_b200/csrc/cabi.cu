// extern "C" surface of libmpe_b200.so (declared in include/mpe_b200.h).  Handles, argument
// checking, error text; all compute is in the kernel translation units behind env_launch.h /
// actor_launch.h.  No host synchronisation except where the header says so.
#include <cuda_runtime.h>

#include <cstdio>
#include <cstring>
#include <new>
#include <string>

#include "../../include/mpe_b200.h"
#include "actor_launch.h"
#include "critic_launch.h"
#include "env_launch.h"
#include "launch.h"
#include "replay_launch.h"

namespace {

thread_local std::string g_err;

int fail(int code, const std::string &msg) {
  g_err = msg;
  return code;
}
int fail_cuda(cudaError_t e, const char *where) {
  g_err = std::string(where) + ": " + cudaGetErrorName(e) + " (" + cudaGetErrorString(e) + ")";
  return MPE_ECUDA;
}

#define CK(call)                                         \
  do {                                                   \
    cudaError_t e_ = (call);                             \
    if (e_ != cudaSuccess) return fail_cuda(e_, #call);  \
  } while (0)

struct DeviceGuard {
  int prev = -1;
  bool ok = true, switched = false;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
    if (prev != dev) {
      if (cudaSetDevice(dev) != cudaSuccess) ok = false; else switched = true;
    }
  }
  ~DeviceGuard() {
    if (switched) cudaSetDevice(prev);  // the common case - already on the handle's device - costs one cudaGetDevice
  }
};

size_t real_size(int precision) { return precision == MPE_F64 ? sizeof(double) : sizeof(float); }

}  // namespace

struct MpeEnv {
  mpe::EnvStateAny st;
  int device = 0;
  // lazily allocated device mirrors for the *_host entry points
  int32_t *h_act_u = nullptr, *h_act_c = nullptr;
  void *h_obs = nullptr, *h_rew = nullptr;
  uint8_t *h_done = nullptr;
  // scratch of the per-step rollout (teams of > 3 agents, the FFMA actor): current observations and sampled actions
  float *r_obs = nullptr;
  int32_t *r_act = nullptr;
  // mpe_rollout_replay: the per-step path's second observation buffer (obs_t and obs_{t+1} of one transition must
  // both survive the step) and rewards when the caller records none; the fused path's recordings of one segment
  float *r_obs2 = nullptr, *r_rew = nullptr;
  unsigned char *rr_scratch = nullptr;
  size_t rr_bytes = 0;
  // mpe_act_step_host_async: device mirror of the caller's observations and of its transition block
  float *hb_obs_in = nullptr;
  unsigned char *hb_block = nullptr;
  // dense2-share scratch of the tensor-core actor for launches made on THIS env's stream (mpe_rollout's per-step path,
  // mpe_act_step_host_async): several env shards share one actor handle on different streams (HostRollout), and the
  // large-team / two-head actor kernels park partial logits in a scratch buffer - one per stream, not one per actor
  float *tc_scratch = nullptr;
  bool synced = false;      // all envs are at the same episode step (true after an unmasked reset)
  int32_t host_tstep = 0;   // that common episode step
};

struct ActorMirror {
  float *obs = nullptr, *onehot = nullptr;  // device mirrors for actor_forward_host
  int32_t *act_u = nullptr, *act_c = nullptr;
  int64_t cap = 0;  // capacity in rows (B*N)
};

struct MpeActor {
  mpe::ActorDev dev;
  int device = 0;
  float *stage = nullptr;  // actor_load: device copy of the caller's host tensors, read by the pack kernel
  ActorMirror mirror;
  float *hcat = nullptr;  // [rows][64] relu(BiLSTM output) between the tensor-core forward and the dense3 head
  int64_t hcat_rows = 0;
};

struct MpeCritic {
  mpe::CriticDev dev;
  int device = 0;
  float *stage = nullptr;  // critic_load: device copy of the caller's host tensors, read by the pack kernel
};

struct MpeReplay {
  mpe::ReplayDev dev;
  int device = 0;
  int64_t size = 0, head = 0;  // host-side ring counters (rls/replay_buffer.py: len(_storage), _next_idx)
  uint64_t draws = 0;          // Philox counter of make_index calls
  int64_t *idx_scratch = nullptr;  // indices drawn by replay_sample when the caller passes none
  int64_t idx_cap = 0;
};

static cudaError_t ensure_tc_scratch(float **p, int device) {
  if (*p != nullptr) return cudaSuccess;
  return cudaMalloc(p, mpe::tc_scratch_floats(mpe::sm_count(device)) * sizeof(float));
}

// The actor's tensor-core weights for a launch on the caller's stream.  The kernels of large teams (N > 3) and of
// two-head actors write per-cell logits shares to a scratch buffer indexed by CTA: two launches in flight on
// different streams must not share it, so a caller that passes `stream_scratch` gets that buffer (allocated on first
// use) instead of the actor's own.
static cudaError_t tc_for_stream(const MpeActor *a, int N, float **stream_scratch, mpe::TcDev *out) {
  *out = a->dev.tc;
  if (stream_scratch == nullptr || (N <= 3 && a->dev.tc.A <= 8)) return cudaSuccess;
  cudaError_t e = ensure_tc_scratch(stream_scratch, a->device);
  out->scratch = *stream_scratch;
  return e;
}

static bool use_tc(const MpeActor *a, int N) {
  return a->dev.impl != mpe::kImplSimt && mpe::tc_actor_supported(a->dev.tc, N);
}

// One actor forward on `st`: tensor cores where they cover the shape, else the fp32 FFMA kernel.
static cudaError_t launch_actor(const MpeActor *a, const mpe::ActorIO &io, float **stream_scratch, cudaStream_t st) {
  if (!use_tc(a, io.N)) return mpe::launch_actor_forward(a->dev, io, st);
  mpe::TcDev tc;
  cudaError_t e = tc_for_stream(a, io.N, stream_scratch, &tc);
  return e != cudaSuccess ? e : mpe::launch_actor_forward_tc(tc, io, st);
}

// The weight structs field by field, with the element count of the reference tensor behind each field for a handle
// (0: the handle does not read that field).
constexpr int kActorFields = 16, kCriticFields = 10;
static const float *ActorWeights::*const kActorField[kActorFields] = {
    &ActorWeights::dense1_w, &ActorWeights::dense1_b, &ActorWeights::w_ih,     &ActorWeights::w_hh,
    &ActorWeights::b_ih,     &ActorWeights::b_hh,     &ActorWeights::w_ih_r,   &ActorWeights::w_hh_r,
    &ActorWeights::b_ih_r,   &ActorWeights::b_hh_r,   &ActorWeights::dense2_w, &ActorWeights::dense2_b,
    &ActorWeights::dense2b_w, &ActorWeights::dense2b_b, &ActorWeights::dense3_w, &ActorWeights::dense3_b};
static const float *CriticWeights::*const kCriticField[kCriticFields] = {
    &CriticWeights::dense1_w, &CriticWeights::dense1_b, &CriticWeights::w_ih,     &CriticWeights::w_hh,
    &CriticWeights::b_ih,     &CriticWeights::b_hh,     &CriticWeights::dense2_w, &CriticWeights::dense2_b,
    &CriticWeights::dense3_w, &CriticWeights::dense3_b};

static void actor_counts(const mpe::ActorDev &d, size_t (&n)[kActorFields]) {
  const size_t H = mpe::kHid, G = mpe::kGateN, D = d.D, A0 = d.A0, A1 = d.A1, M = d.has_model ? 1 : 0;
  const size_t c[kActorFields] = {H * D, H, G * H, G * mpe::kH, G, G, G * H, G * mpe::kH, G, G,
                                  A0 * H, A0, A1 * H, A1, M * D * H, M * D};
  for (int f = 0; f < kActorFields; ++f) n[f] = c[f];
}
static void critic_counts(const mpe::CriticDev &d, size_t (&n)[kCriticFields]) {
  const size_t H = mpe::kCriticH, G = 4 * mpe::kCriticH, Din = d.Din, O = d.out, R = d.has_r ? 1 : 0;
  const size_t c[kCriticFields] = {H * Din, H, G * H, G * H, G, G, O * H, O, R * O * H, R * O};
  for (int f = 0; f < kCriticFields; ++f) n[f] = c[f];
}
template <int F>
static size_t total(const size_t (&n)[F]) {
  size_t t = 0;
  for (int f = 0; f < F; ++f) t += n[f];
  return t;
}

// Device or managed memory of `device`.  A host pointer - pageable, pinned or registered - is refused.
static bool device_memory(const void *p, int device) {
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
    cudaGetLastError();  // not a pointer the runtime knows: do not leave the error for the caller's next check
    return false;
  }
  return (at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged) && at.device == device;
}

// device mirrors of the mpe_*_host entry points, allocated on first use
static cudaError_t ensure_host_mirrors(MpeEnv *env) {
  const mpe::EnvStateAny &s = env->st;
  const size_t rows = (size_t)s.B * s.N, rs = real_size(s.precision);
  cudaError_t e = cudaSuccess;
  auto alloc = [&](auto **p, size_t bytes) {
    if (e == cudaSuccess && *p == nullptr) e = cudaMalloc(p, bytes);
  };
  alloc(&env->h_act_u, rows * sizeof(int32_t));
  alloc(&env->h_act_c, rows * sizeof(int32_t));
  alloc(&env->h_obs, rows * s.D * rs);
  alloc(&env->h_rew, rows * rs);
  alloc(&env->h_done, rows);
  return e;
}

extern "C" {

int mpe_abi_version(void) { return MPE_ABI_VERSION; }
const char *mpe_last_error(void) { return g_err.c_str(); }

int mpe_create(const MpeConfig *cfg, MpeEnv **out) {
  if (cfg == nullptr || out == nullptr) return fail(MPE_EINVAL, "mpe_create: null argument");
  *out = nullptr;
  if (cfg->num_envs <= 0) return fail(MPE_EINVAL, "mpe_create: num_envs must be > 0");
  if (cfg->precision != MPE_F32 && cfg->precision != MPE_F64) return fail(MPE_EINVAL, "mpe_create: bad precision");
  int N = cfg->num_agents, L, D, dimc, act_c = 0;
  switch (cfg->scenario) {
    case MPE_SIMPLE_SPREAD:
      if (N == 0) N = 3;
      L = N; D = 4 + 2 * L; dimc = 2;
      break;
    case MPE_SIMPLE_REFERENCE:
      if (N != 0 && N != 2) return fail(MPE_EUNSUPPORTED, "simple_reference has exactly 2 agents");
      N = 2; L = 3; D = 21; dimc = 10; act_c = 10;
      break;
    case MPE_SIMPLE_SPEAKER_LISTENER:
      if (N != 0 && N != 2) return fail(MPE_EUNSUPPORTED, "simple_speaker_listener has exactly 2 agents");
      N = 2; L = 3; D = 11; dimc = 3;
      break;
    case MPE_COLLECT_TREASURE:  // MAAC fork: make_world() takes no agent count (8 agents: 6 collectors + 2 deposits)
      if (N != 0 && N != 8) return fail(MPE_EUNSUPPORTED, "fullobs_collect_treasure has exactly 8 agents");
      N = 8; L = 6; D = 30; dimc = 2;
      break;
    default:
      return fail(MPE_EUNSUPPORTED, "mpe_create: unknown scenario");
  }
  if (!mpe::env_supported(cfg->scenario, N)) {
    char buf[128];
    snprintf(buf, sizeof buf, "mpe_create: no kernel instantiated for scenario %d with %d agents", cfg->scenario, N);
    return fail(MPE_EUNSUPPORTED, buf);
  }
  DeviceGuard g(cfg->device);
  if (!g.ok) return fail(MPE_ECUDA, "mpe_create: cannot select device");
  MpeEnv *env = new (std::nothrow) MpeEnv();
  if (env == nullptr) return fail(MPE_EINVAL, "mpe_create: out of host memory");
  env->device = cfg->device;
  mpe::EnvStateAny &s = env->st;
  s.B = cfg->num_envs; s.gid0 = cfg->env_id_offset; s.seed = cfg->seed;
  s.max_speed = cfg->max_speed; s.accel = cfg->accel;
  if (cfg->scenario == MPE_COLLECT_TREASURE) {  // the scenario sets accel = 1.5 and max_speed = 1.0 on every agent
    if (s.max_speed < 0.0) s.max_speed = 1.0;
    if (s.accel < 0.0) s.accel = 1.5;
  }
  s.precision = cfg->precision; s.scenario = cfg->scenario;
  s.N = N; s.L = L; s.D = D; s.dimc = dimc; s.act_u = 5; s.act_c = act_c;
  s.max_episode_len = cfg->max_episode_len > 0 ? cfg->max_episode_len : 0;
  const size_t rs = real_size(cfg->precision);
  const size_t B = (size_t)s.B;
  cudaError_t e = cudaSuccess;
  auto alloc = [&](void **p, size_t bytes, int fill) {
    if (e != cudaSuccess) return;
    e = cudaMalloc(p, bytes);
    if (e == cudaSuccess) e = cudaMemset(*p, fill, bytes);
  };
  alloc(&s.pv, (size_t)N * B * 4 * rs, 0);
  alloc(&s.lm, (size_t)L * B * 2 * rs, 0);
  alloc(&s.ep_ret, B * rs, 0);
  alloc(reinterpret_cast<void **>(&s.goal), B * sizeof(int32_t), 0xFF);
  alloc(reinterpret_cast<void **>(&s.episode), B * sizeof(uint32_t), 0xFF);  // first reset -> episode 0
  alloc(reinterpret_cast<void **>(&s.tstep), B * sizeof(int32_t), 0);
  alloc(reinterpret_cast<void **>(&s.stats), 8 * sizeof(double), 0);  // MPE_STATS_LEN used, padded to 64 B
  if (cfg->scenario == MPE_SIMPLE_REFERENCE) alloc(&s.comm, (size_t)N * dimc * B * rs, 0);
  if (e != cudaSuccess) {
    mpe_destroy(env);
    return fail_cuda(e, "mpe_create: cudaMalloc");
  }
  *out = env;
  return MPE_OK;
}

int mpe_destroy(MpeEnv *env) {
  if (env == nullptr) return MPE_OK;
  DeviceGuard g(env->device);
  cudaDeviceSynchronize();
  mpe::EnvStateAny &s = env->st;
  void *ptrs[] = {s.pv, s.lm, s.ep_ret, s.comm, s.goal, s.episode, s.tstep, s.stats,
                  env->h_act_u, env->h_act_c, env->h_obs, env->h_rew, env->h_done, env->r_obs, env->r_act,
                  env->r_obs2, env->r_rew, env->rr_scratch, env->hb_obs_in, env->hb_block, env->tc_scratch};
  for (void *p : ptrs)
    if (p != nullptr) cudaFree(p);
  delete env;
  return MPE_OK;
}

int mpe_query(const MpeEnv *env, MpeDims *out) {
  if (env == nullptr || out == nullptr) return fail(MPE_EINVAL, "mpe_query: null argument");
  const mpe::EnvStateAny &s = env->st;
  out->num_agents = s.N; out->num_landmarks = s.L; out->obs_dim = s.D; out->dim_c = s.dimc;
  out->act_u = s.act_u; out->act_c = s.act_c; out->precision = s.precision; out->device = env->device;
  out->num_envs = s.B; out->env_id_offset = s.gid0;
  return MPE_OK;
}

int mpe_seed(MpeEnv *env, uint64_t seed, void *stream) {
  if (env == nullptr) return fail(MPE_EINVAL, "mpe_seed: null env");
  DeviceGuard g(env->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  mpe::EnvStateAny &s = env->st;
  s.seed = seed;
  // restart the episode counters so that (seed, env id, episode) streams are reproducible, and drop the
  // half-finished episodes' bookkeeping (the next reset starts episode 0 of the new seed)
  CK(cudaMemsetAsync(s.episode, 0xFF, (size_t)s.B * sizeof(uint32_t), st));
  CK(cudaMemsetAsync(s.tstep, 0, (size_t)s.B * sizeof(int32_t), st));
  CK(cudaMemsetAsync(s.ep_ret, 0, (size_t)s.B * real_size(s.precision), st));
  env->synced = false;
  env->host_tstep = 0;
  return MPE_OK;
}

int mpe_reset(MpeEnv *env, const uint8_t *mask, void *obs_out, void *stream) {
  if (env == nullptr) return fail(MPE_EINVAL, "mpe_reset: null env");
  DeviceGuard g(env->device);
  CK(mpe::launch_reset(env->st, mask, obs_out, 0, static_cast<cudaStream_t>(stream)));
  env->synced = mask == nullptr;  // every env starts an episode together
  env->host_tstep = mask == nullptr ? 0 : env->host_tstep;
  return MPE_OK;
}

int mpe_set_state(MpeEnv *env, const void *pos, const void *vel, const void *lm, const int32_t *goal, void *stream) {
  if (env == nullptr) return fail(MPE_EINVAL, "mpe_set_state: null env");
  DeviceGuard g(env->device);
  CK(mpe::launch_set_state(env->st, pos, vel, lm, goal, static_cast<cudaStream_t>(stream)));
  env->synced = false;
  return MPE_OK;
}

int mpe_get_state(MpeEnv *env, void *pos, void *vel, void *lm, int32_t *goal, void *stream) {
  if (env == nullptr) return fail(MPE_EINVAL, "mpe_get_state: null env");
  DeviceGuard g(env->device);
  CK(mpe::launch_get_state(env->st, pos, vel, lm, goal, static_cast<cudaStream_t>(stream)));
  return MPE_OK;
}

int mpe_observe(MpeEnv *env, void *obs_out, void *stream) {
  if (env == nullptr || obs_out == nullptr) return fail(MPE_EINVAL, "mpe_observe: null argument");
  DeviceGuard g(env->device);
  CK(mpe::launch_observe(env->st, obs_out, static_cast<cudaStream_t>(stream)));
  return MPE_OK;
}

int mpe_step(MpeEnv *env, const int32_t *act_u, const int32_t *act_c, const void *comm_vec, void *obs, void *rew,
             uint8_t *done, int32_t *info_i, void *info_f, void *stream) {
  if (env == nullptr || act_u == nullptr) return fail(MPE_EINVAL, "mpe_step: null env or act_u");
  if (env->st.scenario == MPE_SIMPLE_REFERENCE && act_c == nullptr && comm_vec == nullptr)
    return fail(MPE_EINVAL, "mpe_step: simple_reference needs act_c or comm_vec");
  DeviceGuard g(env->device);
  CK(mpe::launch_step(env->st, act_u, act_c, comm_vec, obs, rew, done, info_i, info_f,
                      static_cast<cudaStream_t>(stream)));
  if (env->st.track) env->host_tstep += 1; else env->synced = false;
  return MPE_OK;
}

int mpe_step_host(MpeEnv *env, const int32_t *act_u_host, const int32_t *act_c_host, void *obs_host, void *rew_host,
                  uint8_t *done_host, void *stream) {
  if (env == nullptr || act_u_host == nullptr) return fail(MPE_EINVAL, "mpe_step_host: null env or act_u");
  if (env->st.scenario == MPE_SIMPLE_REFERENCE && act_c_host == nullptr)
    return fail(MPE_EINVAL, "mpe_step_host: simple_reference needs act_c");
  DeviceGuard g(env->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const mpe::EnvStateAny &s = env->st;
  const size_t rows = (size_t)s.B * s.N, rs = real_size(s.precision);
  CK(ensure_host_mirrors(env));
  CK(cudaMemcpyAsync(env->h_act_u, act_u_host, rows * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  if (act_c_host != nullptr)
    CK(cudaMemcpyAsync(env->h_act_c, act_c_host, rows * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  CK(mpe::launch_step(s, env->h_act_u, act_c_host != nullptr ? env->h_act_c : nullptr, nullptr,
                      obs_host != nullptr ? env->h_obs : nullptr, rew_host != nullptr ? env->h_rew : nullptr,
                      done_host != nullptr ? env->h_done : nullptr, nullptr, nullptr, st));
  if (env->st.track) env->host_tstep += 1; else env->synced = false;
  if (obs_host != nullptr) CK(cudaMemcpyAsync(obs_host, env->h_obs, rows * s.D * rs, cudaMemcpyDeviceToHost, st));
  if (rew_host != nullptr) CK(cudaMemcpyAsync(rew_host, env->h_rew, rows * rs, cudaMemcpyDeviceToHost, st));
  if (done_host != nullptr) CK(cudaMemcpyAsync(done_host, env->h_done, rows, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return MPE_OK;
}

int mpe_reset_host_async(MpeEnv *env, void *obs_host, void *stream) {
  if (env == nullptr || obs_host == nullptr) return fail(MPE_EINVAL, "mpe_reset_host_async: null argument");
  DeviceGuard g(env->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const mpe::EnvStateAny &s = env->st;
  const size_t rows = (size_t)s.B * s.N, rs = real_size(s.precision);
  CK(ensure_host_mirrors(env));
  CK(mpe::launch_reset(s, nullptr, env->h_obs, 0, st));
  env->synced = true;
  env->host_tstep = 0;
  CK(cudaMemcpyAsync(obs_host, env->h_obs, rows * s.D * rs, cudaMemcpyDeviceToHost, st));
  return MPE_OK;
}

int mpe_track_returns(MpeEnv *env, int32_t enable) {
  if (env == nullptr) return fail(MPE_EINVAL, "mpe_track_returns: null env");
  env->st.track = enable ? 1 : 0;
  return MPE_OK;
}

int mpe_stats_read(MpeEnv *env, double out[MPE_STATS_LEN], int32_t clear, void *stream) {
  if (env == nullptr || out == nullptr) return fail(MPE_EINVAL, "mpe_stats_read: null argument");
  DeviceGuard g(env->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CK(cudaMemcpyAsync(out, env->st.stats, MPE_STATS_LEN * sizeof(double), cudaMemcpyDeviceToHost, st));
  if (clear) CK(cudaMemsetAsync(env->st.stats, 0, MPE_STATS_LEN * sizeof(double), st));
  CK(cudaStreamSynchronize(st));
  return MPE_OK;
}

int mpe_stats_ptr(MpeEnv *env, double **dev_ptr) {
  if (env == nullptr || dev_ptr == nullptr) return fail(MPE_EINVAL, "mpe_stats_ptr: null argument");
  *dev_ptr = env->st.stats;
  return MPE_OK;
}

// ------------------------------------------------------------------------------------------------
// actor
// ------------------------------------------------------------------------------------------------
int actor_destroy(MpeActor *a);

int actor_create(const ActorConfig *cfg, MpeActor **out) {
  if (cfg == nullptr || out == nullptr) return fail(MPE_EINVAL, "actor_create: null argument");
  *out = nullptr;
  if (cfg->obs_dim <= 0 || cfg->obs_dim > mpe::kActorMaxD) return fail(MPE_EUNSUPPORTED, "actor_create: obs_dim out of range");
  if (cfg->act0 <= 0 || cfg->act1 < 0 || cfg->act0 + cfg->act1 > mpe::kActorMaxA)
    return fail(MPE_EUNSUPPORTED, "actor_create: head widths out of range");
  DeviceGuard g(cfg->device);
  if (!g.ok) return fail(MPE_ECUDA, "actor_create: cannot select device");
  MpeActor *a = new (std::nothrow) MpeActor();
  if (a == nullptr) return fail(MPE_EINVAL, "actor_create: out of host memory");
  a->device = cfg->device;
  mpe::actor_layout(cfg->obs_dim, cfg->act0, cfg->act1, cfg->has_model_head != 0, &a->dev);
  mpe::tc_layout(cfg->obs_dim, cfg->act0, cfg->act1, &a->dev.tc);
  cudaError_t e = cudaMalloc(&a->dev.blob, a->dev.blob_floats * sizeof(float));
  if (e == cudaSuccess) e = cudaMemset(a->dev.blob, 0, a->dev.blob_floats * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc(&a->dev.tc.blob, a->dev.tc.bytes);
  if (e == cudaSuccess) e = cudaMemset(a->dev.tc.blob, 0, a->dev.tc.bytes);
  if (e == cudaSuccess) e = ensure_tc_scratch(&a->dev.tc.scratch, cfg->device);
  size_t n[kActorFields];
  actor_counts(a->dev, n);
  if (e == cudaSuccess) e = cudaMalloc(&a->stage, total(n) * sizeof(float));
  if (e != cudaSuccess) {
    actor_destroy(a);  // frees whatever was allocated before the failure
    return fail_cuda(e, "actor_create: cudaMalloc");
  }
  *out = a;
  return MPE_OK;
}

int actor_destroy(MpeActor *a) {
  if (a == nullptr) return MPE_OK;
  DeviceGuard g(a->device);
  cudaDeviceSynchronize();
  void *ptrs[] = {a->dev.blob, a->dev.tc.blob, a->dev.tc.scratch, a->hcat, a->stage};
  for (void *p : ptrs)
    if (p != nullptr) cudaFree(p);
  const ActorMirror &m = a->mirror;
  void *mp[] = {m.obs, m.onehot, m.act_u, m.act_c};
  for (void *p : mp)
    if (p != nullptr) cudaFree(p);
  delete a;
  return MPE_OK;
}

static int check_actor_weights(const MpeActor *a, const ActorWeights *w, const char *who) {
  const std::string n(who);
  if (a == nullptr || w == nullptr) return fail(MPE_EINVAL, n + ": null argument");
  if (!w->dense1_w || !w->dense1_b || !w->w_ih || !w->w_hh || !w->b_ih || !w->b_hh || !w->w_ih_r || !w->w_hh_r ||
      !w->b_ih_r || !w->b_hh_r || !w->dense2_w || !w->dense2_b)
    return fail(MPE_EINVAL, n + ": missing tensor");
  if (a->dev.A1 > 0 && (!w->dense2b_w || !w->dense2b_b)) return fail(MPE_EINVAL, n + ": missing dense2_2");
  if (a->dev.has_model && (!w->dense3_w || !w->dense3_b)) return fail(MPE_EINVAL, n + ": missing dense3");
  return MPE_OK;
}

// The host tensors are copied into the handle's staging buffer and packed by the same kernel as actor_load_device;
// the synchronise frees both the caller's arrays and the staging buffer.
int actor_load(MpeActor *a, const ActorWeights *w, void *stream) {
  if (int rc = check_actor_weights(a, w, "actor_load")) return rc;
  DeviceGuard g(a->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  size_t n[kActorFields];
  actor_counts(a->dev, n);
  ActorWeights staged = {};
  float *p = a->stage;
  for (int f = 0; f < kActorFields; ++f) {
    if (n[f] == 0) continue;
    CK(cudaMemcpyAsync(p, w->*kActorField[f], n[f] * sizeof(float), cudaMemcpyHostToDevice, st));
    staged.*kActorField[f] = p;
    p += n[f];
  }
  CK(mpe::launch_actor_pack(a->dev, staged, st));
  CK(cudaStreamSynchronize(st));
  return MPE_OK;
}

int actor_load_device(MpeActor *a, const ActorWeights *w, void *stream) {
  if (int rc = check_actor_weights(a, w, "actor_load_device")) return rc;
  size_t n[kActorFields];
  actor_counts(a->dev, n);
  ActorWeights src = {};  // the fields this actor reads; the rest stay NULL
  for (int f = 0; f < kActorFields; ++f) {
    if (n[f] == 0) continue;
    if (!device_memory(w->*kActorField[f], a->device))
      return fail(MPE_EINVAL, "actor_load_device: a weight pointer is not device memory on the actor's device");
    src.*kActorField[f] = w->*kActorField[f];
  }
  DeviceGuard g(a->device);
  CK(mpe::launch_actor_pack(a->dev, src, static_cast<cudaStream_t>(stream)));
  return MPE_OK;
}

int actor_set_impl(MpeActor *a, int32_t impl) {
  if (a == nullptr || impl < mpe::kImplAuto || impl > mpe::kImplTc) return fail(MPE_EINVAL, "actor_set_impl: bad argument");
  a->dev.impl = impl;
  return MPE_OK;
}

int actor_forward(MpeActor *a, const float *obs, int64_t B, int32_t N, const float *gumbel, uint64_t seed,
                  uint64_t step, int64_t env_id_offset, float *logits, float *next_state, int32_t *act_u,
                  int32_t *act_c, float *onehot, void *stream) {
  if (a == nullptr || obs == nullptr) return fail(MPE_EINVAL, "actor_forward: null argument");
  if (B <= 0) return MPE_OK;
  if (!mpe::actor_supported(N)) return fail(MPE_EUNSUPPORTED, "actor_forward: unsupported agent count");
  if (next_state != nullptr && !a->dev.has_model) return fail(MPE_EINVAL, "actor_forward: no model head loaded");
  DeviceGuard g(a->device);
  mpe::ActorIO io;
  io.obs = obs; io.gumbel = gumbel; io.logits = logits; io.next_state = next_state;
  io.act_u = act_u; io.act_c = act_c; io.onehot = onehot;
  io.B = B; io.N = N; io.seed = seed; io.step = step; io.gid0 = env_id_offset;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bool tc = use_tc(a, N);
  if (a->dev.impl == mpe::kImplTc && !tc)
    return fail(MPE_EUNSUPPORTED, "actor_forward: the tensor-core path covers 2/3/4/6/8/9/12 agents, obs_dim <= 32, <= 8 head entries for > 3 agents");
  if (tc && next_state != nullptr) {  // "+model" head: the forward leaves relu(hcat) behind, one small kernel applies dense3
    const int64_t rows = B * N;
    if (rows > a->hcat_rows) {
      if (a->hcat != nullptr) { CK(cudaStreamSynchronize(st)); cudaFree(a->hcat); a->hcat = nullptr; a->hcat_rows = 0; }
      CK(cudaMalloc(&a->hcat, (size_t)rows * 64 * sizeof(float)));
      a->hcat_rows = rows;
    }
    io.hcat = a->hcat;
    io.next_state = nullptr;
  }
  CK(launch_actor(a, io, nullptr, st));
  if (io.hcat != nullptr) CK(mpe::launch_dense3(a->dev, a->hcat, B * N, next_state, st));
  return MPE_OK;
}

// H2D obs -> forward + sample -> D2H actions, all enqueued on `stream`, then a stream synchronise.
int actor_forward_host(MpeActor *a, const float *obs_host, int64_t B, int32_t N, uint64_t seed, uint64_t step,
                       int64_t env_id_offset, int32_t *act_u_host, int32_t *act_c_host, float *onehot_host,
                       void *stream) {
  if (a == nullptr || obs_host == nullptr) return fail(MPE_EINVAL, "actor_forward_host: null argument");
  if (B <= 0) return MPE_OK;
  if (!mpe::actor_supported(N)) return fail(MPE_EUNSUPPORTED, "actor_forward_host: unsupported agent count");
  DeviceGuard g(a->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t rows = B * N;
  const int A = a->dev.A0 + a->dev.A1;
  ActorMirror &m = a->mirror;
  if (rows > m.cap) {
    // growing the mirror frees the old one: wait for whatever the stream still has in flight on it
    if (m.cap > 0) CK(cudaStreamSynchronize(st));
    void *old[] = {m.obs, m.onehot, m.act_u, m.act_c};
    for (void *p : old)
      if (p != nullptr) cudaFree(p);
    m = ActorMirror();
    CK(cudaMalloc(&m.obs, (size_t)rows * a->dev.D * sizeof(float)));
    CK(cudaMalloc(&m.onehot, (size_t)rows * A * sizeof(float)));
    CK(cudaMalloc(&m.act_u, (size_t)rows * sizeof(int32_t)));
    CK(cudaMalloc(&m.act_c, (size_t)rows * sizeof(int32_t)));
    m.cap = rows;
  }
  CK(cudaMemcpyAsync(m.obs, obs_host, (size_t)rows * a->dev.D * sizeof(float), cudaMemcpyHostToDevice, st));
  mpe::ActorIO io;
  io.obs = m.obs; io.act_u = m.act_u; io.act_c = a->dev.A1 > 0 ? m.act_c : nullptr;
  io.onehot = onehot_host != nullptr ? m.onehot : nullptr;
  io.B = B; io.N = N; io.seed = seed; io.step = step; io.gid0 = env_id_offset;
  CK(launch_actor(a, io, nullptr, st));
  if (act_u_host != nullptr) CK(cudaMemcpyAsync(act_u_host, m.act_u, (size_t)rows * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  if (act_c_host != nullptr && a->dev.A1 > 0)
    CK(cudaMemcpyAsync(act_c_host, m.act_c, (size_t)rows * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  if (onehot_host != nullptr)
    CK(cudaMemcpyAsync(onehot_host, m.onehot, (size_t)rows * A * sizeof(float), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return MPE_OK;
}

int64_t actor_backward_workspace(MpeActor *a, int64_t B, int32_t N) {
  if (a == nullptr) return fail(MPE_EINVAL, "actor_backward_workspace: null actor");
  if (B < 0) return fail(MPE_EINVAL, "actor_backward_workspace: B < 0");
  if (!mpe::actor_supported(N)) return fail(MPE_EUNSUPPORTED, "actor_backward_workspace: 1..12 agents");
  return mpe::actor_backward_bytes(a->dev, B, N);
}

int actor_backward(MpeActor *a, const float *obs, int64_t B, int32_t N, const float *dlogits, const float *dnext_state,
                   float *dobs, const ActorGrads *grads, void *workspace, int64_t workspace_bytes, void *stream) {
  if (a == nullptr || obs == nullptr || dlogits == nullptr || workspace == nullptr)
    return fail(MPE_EINVAL, "actor_backward: null argument");
  if (B < 0) return fail(MPE_EINVAL, "actor_backward: B < 0");
  if (!mpe::actor_supported(N)) return fail(MPE_EUNSUPPORTED, "actor_backward: 1..12 agents");
  const ActorGrads none = {};
  const ActorGrads &g = grads != nullptr ? *grads : none;
  if (!a->dev.has_model && (dnext_state != nullptr || g.dense3_w != nullptr || g.dense3_b != nullptr))
    return fail(MPE_EINVAL, "actor_backward: dnext_state / dense3 gradients on an actor without a model head");
  if (a->dev.A1 == 0 && (g.dense2b_w != nullptr || g.dense2b_b != nullptr))
    return fail(MPE_EINVAL, "actor_backward: dense2_2 gradients on a single-head actor");
  const int64_t need = mpe::actor_backward_bytes(a->dev, B, N);
  if (workspace_bytes < need)
    return fail(MPE_EINVAL, "actor_backward: workspace of " + std::to_string(workspace_bytes) + " bytes, " +
                                std::to_string(need) + " needed");
  if (B == 0) return MPE_OK;
  const void *ptrs[] = {obs, dlogits, dnext_state, dobs, workspace, g.dense1_w, g.dense1_b, g.w_ih, g.w_hh, g.b_ih,
                        g.b_hh, g.w_ih_r, g.w_hh_r, g.b_ih_r, g.b_hh_r, g.dense2_w, g.dense2_b, g.dense2b_w,
                        g.dense2b_b, g.dense3_w, g.dense3_b};
  for (const void *p : ptrs)
    if (p != nullptr && !device_memory(p, a->device))
      return fail(MPE_EINVAL, "actor_backward: a pointer is not device memory on the actor's device");
  DeviceGuard dg(a->device);
  CK(mpe::launch_actor_backward(a->dev, obs, B, N, dlogits, dnext_state, dobs, g, workspace,
                                static_cast<cudaStream_t>(stream)));
  return MPE_OK;
}

static MpeHostBlockLayout block_layout(const mpe::EnvStateAny &s) {
  const uint64_t rows = (uint64_t)s.B * s.N, rs = real_size(s.precision);
  auto up = [](uint64_t x) { return (x + 255) / 256 * 256; };
  MpeHostBlockLayout l;
  l.off_act_u = 0;
  l.off_act_c = up(l.off_act_u + rows * 4);
  l.off_obs = up(l.off_act_c + (s.act_c > 0 ? rows * 4 : 0));  // no message head: act_c has zero length (off_act_c == off_obs)
  l.off_rew = up(l.off_obs + rows * s.D * rs);
  l.off_done = up(l.off_rew + rows * rs);
  l.bytes = up(l.off_done + rows);
  return l;
}

int mpe_host_block_layout(const MpeEnv *env, MpeHostBlockLayout *out) {
  if (env == nullptr || out == nullptr) return fail(MPE_EINVAL, "mpe_host_block_layout: null argument");
  *out = block_layout(env->st);
  return MPE_OK;
}

int mpe_act_step_host_async(MpeEnv *env, MpeActor *actor, const float *obs_host, uint64_t step, void *block_host,
                            void *stream) {
  if (env == nullptr || actor == nullptr || obs_host == nullptr || block_host == nullptr)
    return fail(MPE_EINVAL, "mpe_act_step_host_async: null argument");
  mpe::EnvStateAny &s = env->st;
  if (s.precision != MPE_F32) return fail(MPE_EUNSUPPORTED, "mpe_act_step_host_async: fp32 envs only");
  if (env->device != actor->device) return fail(MPE_EINVAL, "mpe_act_step_host_async: env and actor on different devices");
  if (actor->dev.D != s.D || actor->dev.A0 != 5 || actor->dev.A1 != s.act_c)
    return fail(MPE_EINVAL, "mpe_act_step_host_async: actor does not match the env's observation / action space");
  if (!mpe::actor_supported(s.N)) return fail(MPE_EUNSUPPORTED, "mpe_act_step_host_async: unsupported agent count");
  DeviceGuard g(env->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const MpeHostBlockLayout l = block_layout(s);
  const size_t rows = (size_t)s.B * s.N;
  if (env->hb_block == nullptr) {
    CK(cudaMalloc(&env->hb_obs_in, rows * s.D * sizeof(float)));
    CK(cudaMalloc(&env->hb_block, l.bytes));
    CK(cudaMemsetAsync(env->hb_block, 0, l.bytes, st));
  }
  unsigned char *blk = env->hb_block;
  CK(cudaMemcpyAsync(env->hb_obs_in, obs_host, rows * s.D * sizeof(float), cudaMemcpyHostToDevice, st));
  mpe::ActorIO io;
  io.obs = env->hb_obs_in;
  io.act_u = reinterpret_cast<int32_t *>(blk + l.off_act_u);
  io.act_c = actor->dev.A1 > 0 ? reinterpret_cast<int32_t *>(blk + l.off_act_c) : nullptr;
  io.B = s.B; io.N = s.N; io.seed = s.seed; io.step = step; io.gid0 = s.gid0;
  CK(launch_actor(actor, io, &env->tc_scratch, st));  // shards share the actor handle on different streams: scratch per env handle
  CK(mpe::launch_step(s, io.act_u, io.act_c, nullptr, blk + l.off_obs, blk + l.off_rew, blk + l.off_done, nullptr, nullptr, st));
  if (s.track) env->host_tstep += 1; else env->synced = false;
  CK(cudaMemcpyAsync(block_host, blk, l.bytes, cudaMemcpyDeviceToHost, st));
  return MPE_OK;
}

int mpe_host_alloc(void **out, uint64_t bytes) {
  if (out == nullptr || bytes == 0) return fail(MPE_EINVAL, "mpe_host_alloc: bad argument");
  *out = nullptr;
  CK(cudaHostAlloc(out, (size_t)bytes, cudaHostAllocDefault));
  return MPE_OK;
}

int mpe_host_free(void *p) {
  if (p != nullptr) CK(cudaFreeHost(p));
  return MPE_OK;
}

int mpe_host_wait(void *stream) {
  CK(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
  return MPE_OK;
}

// The common episode step of a synced env after T fused iterations (every env resets when its step reaches L).
static void advance_episode_step(MpeEnv *env, int64_t T) {
  const int L = env->st.max_episode_len;
  if (!env->synced || L <= 0) return;  // without auto-reset the episode step never decides a launch
  const int64_t first_end = env->host_tstep >= L ? 1 : L - env->host_tstep;
  env->host_tstep = T < first_end ? (int32_t)(env->host_tstep + T) : (int32_t)((T - first_end) % L);
}

static bool use_fused_rollout(const MpeEnv *env, const MpeActor *actor) {
  return actor->dev.impl != mpe::kImplSimt && mpe::tc_rollout_supported(actor->dev.tc, env->st.N);
}

static int check_rollout(const MpeEnv *env, const MpeActor *actor, const char *who) {
  const std::string w(who);
  if (env->st.precision != MPE_F32) return fail(MPE_EUNSUPPORTED, w + ": fp32 envs only");
  if (env->device != actor->device) return fail(MPE_EINVAL, w + ": env and actor on different devices");
  if (actor->dev.D != env->st.D) return fail(MPE_EINVAL, w + ": actor obs_dim does not match the env");
  if (actor->dev.A0 != 5 || actor->dev.A1 != env->st.act_c)
    return fail(MPE_EINVAL, w + ": actor heads do not match the env's action space");
  if (!mpe::rollout_supported(env->st.scenario, env->st.N))
    return fail(MPE_EUNSUPPORTED, w + ": unsupported scenario / agent count");
  return MPE_OK;
}

// Every combination the fused kernel does not cover (teams of > 3 agents, the fp32 FFMA actor, and with a ring envs
// whose episodes are not aligned): the same loop as kernels per step - actor (tensor cores where the shape is covered,
// else FFMA), the env step kernel, and a reset kernel on the steps where an episode can end.  Same Philox keys, same
// arithmetic: bit-identical to the stepwise calls.  With `rep`, each step's B transitions are appended after the step
// and before the reset overwrites the observations: obs_t is `cur`, obs_{t+1} is `o`.
static int rollout_stepwise(MpeEnv *env, MpeActor *actor, MpeReplay *rep, int32_t T, uint64_t step0, float *obs_next,
                            float *rew, int32_t *act_u, int32_t *act_c, int32_t *info_i, float *info_f,
                            cudaStream_t st) {
  mpe::EnvStateAny s = env->st;
  s.track = 1;
  const int64_t rows = s.B * s.N;
  if (env->r_obs == nullptr) {
    CK(cudaMalloc(&env->r_obs, (size_t)rows * s.D * sizeof(float)));
    CK(cudaMalloc(&env->r_act, (size_t)rows * 2 * sizeof(int32_t)));
  }
  if (rep != nullptr && obs_next == nullptr && env->r_obs2 == nullptr)
    CK(cudaMalloc(&env->r_obs2, (size_t)rows * s.D * sizeof(float)));
  if (rep != nullptr && rew == nullptr && env->r_rew == nullptr) CK(cudaMalloc(&env->r_rew, (size_t)rows * sizeof(float)));
  CK(mpe::launch_observe(s, env->r_obs, st));
  const float *cur = env->r_obs;
  const int L = s.max_episode_len;
  for (int t = 0; t < T; ++t) {
    mpe::ActorIO aio;
    aio.obs = cur; aio.B = s.B; aio.N = s.N; aio.seed = s.seed; aio.step = step0 + (uint64_t)t; aio.gid0 = s.gid0;
    aio.act_u = act_u != nullptr ? act_u + (int64_t)t * rows : env->r_act;
    if (s.act_c > 0) aio.act_c = act_c != nullptr ? act_c + (int64_t)t * rows : env->r_act + rows;
    CK(launch_actor(actor, aio, &env->tc_scratch, st));  // rollouts of several envs may share one actor on different streams
    float *o = obs_next != nullptr ? obs_next + (int64_t)t * rows * s.D
                                   : (rep != nullptr && cur == env->r_obs ? env->r_obs2 : env->r_obs);
    float *r = rew != nullptr ? rew + (int64_t)t * rows : (rep != nullptr ? env->r_rew : nullptr);
    int32_t *ii = info_i != nullptr ? info_i + (int64_t)t * s.B * (s.N + 1) : nullptr;
    float *fi = info_f != nullptr ? info_f + (int64_t)t * s.B : nullptr;
    CK(mpe::launch_step(s, aio.act_u, aio.act_c, nullptr, o, r, nullptr, ii, fi, st));
    if (rep != nullptr) {
      CK(mpe::launch_replay_add(rep->dev, rep->head, s.B, cur, aio.act_u, aio.act_c, r, o, nullptr, st));
      rep->head = (rep->head + s.B) % rep->dev.capacity;
      rep->size = rep->size + s.B < rep->dev.capacity ? rep->size + s.B : rep->dev.capacity;
    }
    cur = o;
    env->host_tstep += 1;
    const bool may_end = L > 0 && (!env->synced || env->host_tstep >= L);
    if (may_end) {  // experiments/run.py:59-60; also re-emits the observations the next actor call reads
      CK(mpe::launch_reset(s, nullptr, env->r_obs, L, st));
      cur = env->r_obs;
      if (env->synced) env->host_tstep = 0;
    }
  }
  return MPE_OK;
}

int mpe_rollout(MpeEnv *env, MpeActor *actor, int32_t T, uint64_t step0, float *obs_next, float *rew, int32_t *act_u,
                int32_t *act_c, int32_t *info_i, void *info_f, void *stream) {
  if (env == nullptr || actor == nullptr) return fail(MPE_EINVAL, "mpe_rollout: null handle");
  if (T <= 0) return MPE_OK;
  if (int rc = check_rollout(env, actor, "mpe_rollout")) return rc;
  DeviceGuard g(env->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // One kernel for all T steps: teams of 2 / 3 on the tensor cores (the large teams run faster as actor + step kernels
  // per step, DESIGN.md 4.3)
  if (use_fused_rollout(env, actor)) {
    mpe::RolloutIO io;
    io.T = T; io.step0 = step0; io.obs_next = obs_next; io.rew = rew; io.act_u = act_u; io.act_c = act_c;
    io.info_i = info_i; io.info_f = static_cast<float *>(info_f);
    mpe::TcDev tcw;
    CK(tc_for_stream(actor, env->st.N, &env->tc_scratch, &tcw));  // rollouts of several envs may share one actor
    CK(mpe::launch_rollout_tc(env->st, tcw, io, st));
    advance_episode_step(env, T);
    return MPE_OK;
  }
  return rollout_stepwise(env, actor, nullptr, T, step0, obs_next, rew, act_u, act_c, info_i,
                          static_cast<float *>(info_f), st);
}

// The fused path of mpe_rollout_replay keeps the recordings the caller does not take in an env-owned scratch of at
// most this many bytes, kept until mpe_destroy so that the calls of a training loop do not allocate; a segment is cut
// short where the next step's recordings would not fit (one recorded step of simple_spread N = 3 at 1,048,576 envs is
// 144 MB: 7 steps per segment).
constexpr size_t kRolloutReplayScratchBytes = size_t(1) << 30;

// Synced envs with the fused kernel: the call runs as segments that end at the common episode end (or where the
// scratch is full).  k_tc2 runs each segment unchanged and records into the caller's buffers or the scratch; one
// launch of the multi-step ring writer then builds the segment's records, obs_t of its first step from the
// observation before the segment (mpe_observe after an episode end: the post-reset observation; else a copy of the
// last step's obs_next) and of every later step from the previous step's obs_next.
static int rollout_fused_replay(MpeEnv *env, MpeActor *actor, MpeReplay *rep, int32_t T, uint64_t step0, float *obs_next,
                                float *rew, int32_t *act_u, int32_t *act_c, int32_t *info_i, float *info_f,
                                cudaStream_t st) {
  const mpe::EnvStateAny &s = env->st;
  const int64_t rows = s.B * s.N, obs_step = rows * s.D;
  auto up = [](size_t x) { return (x + 255) / 256 * 256; };
  const size_t b_obs = obs_next ? 0 : up(obs_step * 4), b_rew = rew ? 0 : up(rows * 4), b_au = act_u ? 0 : up(rows * 4),
               b_ac = (act_c || s.act_c == 0) ? 0 : up(rows * 4), per_step = b_obs + b_rew + b_au + b_ac;
  const int L = s.max_episode_len;
  int64_t seg_cap = per_step == 0 ? T : (int64_t)(kRolloutReplayScratchBytes / per_step);
  seg_cap = seg_cap < 1 ? 1 : (seg_cap > T ? T : seg_cap);
  if (L > 0 && seg_cap > L) seg_cap = L;
  if (env->r_obs == nullptr) {
    CK(cudaMalloc(&env->r_obs, (size_t)obs_step * sizeof(float)));
    CK(cudaMalloc(&env->r_act, (size_t)rows * 2 * sizeof(int32_t)));
  }
  const size_t need = per_step * (size_t)seg_cap;
  if (need > env->rr_bytes) {
    if (env->rr_scratch != nullptr) {  // a recording of an earlier call may still be read on this stream
      CK(cudaStreamSynchronize(st));
      cudaFree(env->rr_scratch);
      env->rr_scratch = nullptr; env->rr_bytes = 0;
    }
    CK(cudaMalloc(&env->rr_scratch, need));
    env->rr_bytes = need;
  }
  unsigned char *sc = env->rr_scratch;
  float *sc_obs = reinterpret_cast<float *>(sc);
  float *sc_rew = reinterpret_cast<float *>(sc + b_obs * seg_cap);
  int32_t *sc_au = reinterpret_cast<int32_t *>(sc + (b_obs + b_rew) * seg_cap);
  int32_t *sc_ac = reinterpret_cast<int32_t *>(sc + (b_obs + b_rew + b_au) * seg_cap);
  mpe::TcDev tcw;
  CK(tc_for_stream(actor, s.N, &env->tc_scratch, &tcw));  // rollouts of several envs may share one actor
  const int64_t keep_from = (int64_t)T * s.B - rep->dev.capacity;  // earlier transitions are overwritten in this call
  CK(mpe::launch_observe(s, env->r_obs, st));
  for (int32_t t0 = 0; t0 < T;) {
    int64_t n = T - t0 < seg_cap ? T - t0 : seg_cap;
    const int64_t to_end = L > 0 ? (env->host_tstep >= L ? 1 : L - env->host_tstep) : n;
    if (to_end < n) n = to_end;
    mpe::RolloutIO io;
    io.T = (int32_t)n; io.step0 = step0 + (uint64_t)t0;
    io.obs_next = obs_next ? obs_next + t0 * obs_step : sc_obs;
    io.rew = rew ? rew + t0 * rows : sc_rew;
    io.act_u = act_u ? act_u + t0 * rows : sc_au;
    io.act_c = s.act_c == 0 ? nullptr : (act_c ? act_c + t0 * rows : sc_ac);
    io.info_i = info_i ? info_i + t0 * s.B * (s.N + 1) : nullptr;  // the ring does not read them: no scratch
    io.info_f = info_f ? info_f + t0 * s.B : nullptr;
    CK(mpe::launch_rollout_tc(s, tcw, io, st));
    CK(mpe::launch_replay_add_steps(rep->dev, rep->head, s.B, io.T, (int64_t)t0 * s.B, keep_from, env->r_obs, io.obs_next,
                                    io.act_u, io.act_c, io.rew, st));
    const bool ended = n == to_end && L > 0;
    advance_episode_step(env, n);
    t0 += (int32_t)n;
    if (t0 < T) {
      if (ended) CK(mpe::launch_observe(s, env->r_obs, st));
      else CK(cudaMemcpyAsync(env->r_obs, io.obs_next + (n - 1) * obs_step, (size_t)obs_step * sizeof(float),
                              cudaMemcpyDeviceToDevice, st));
    }
  }
  const int64_t total = (int64_t)T * s.B;
  rep->head = (rep->head + total) % rep->dev.capacity;
  rep->size = rep->size + total < rep->dev.capacity ? rep->size + total : rep->dev.capacity;
  return MPE_OK;
}

int mpe_rollout_replay(MpeEnv *env, MpeActor *actor, MpeReplay *rep, int32_t T, uint64_t step0, float *obs_next,
                       float *rew, int32_t *act_u, int32_t *act_c, int32_t *info_i, void *info_f, void *stream) {
  if (env == nullptr || actor == nullptr || rep == nullptr) return fail(MPE_EINVAL, "mpe_rollout_replay: null handle");
  if (T <= 0) return MPE_OK;
  if (int rc = check_rollout(env, actor, "mpe_rollout_replay")) return rc;
  const mpe::ReplayDev &r = rep->dev;
  if (rep->device != env->device) return fail(MPE_EINVAL, "mpe_rollout_replay: ring and env on different devices");
  if (r.N != env->st.N || r.D != env->st.D)
    return fail(MPE_EINVAL, "mpe_rollout_replay: ring agents / obs_dim do not match the env");
  if (r.A0 != actor->dev.A0 || r.A1 != actor->dev.A1)
    return fail(MPE_EINVAL, "mpe_rollout_replay: ring action heads do not match the actor");
  if (env->st.B > r.capacity) return fail(MPE_EINVAL, "mpe_rollout_replay: batch larger than the ring");
  DeviceGuard g(env->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // the fused kernel needs the episode ends of all envs to coincide: only there can a segment end and the ring
  // writer find every step's obs_t among the recordings
  if (use_fused_rollout(env, actor) && env->synced)
    return rollout_fused_replay(env, actor, rep, T, step0, obs_next, rew, act_u, act_c, info_i,
                                static_cast<float *>(info_f), st);
  return rollout_stepwise(env, actor, rep, T, step0, obs_next, rew, act_u, act_c, info_i, static_cast<float *>(info_f), st);
}

// ------------------------------------------------------------------------------------------------
// critic
// ------------------------------------------------------------------------------------------------
int critic_destroy(MpeCritic *c);

int critic_create(const CriticConfig *cfg, MpeCritic **out) {
  if (cfg == nullptr || out == nullptr) return fail(MPE_EINVAL, "critic_create: null argument");
  *out = nullptr;
  if (cfg->obs_dim <= 0 || cfg->act_dim <= 0 || cfg->obs_dim + cfg->act_dim > mpe::kCriticMaxIn)
    return fail(MPE_EUNSUPPORTED, "critic_create: obs_dim + act_dim out of range");
  if (cfg->out_dim <= 0 || cfg->out_dim > mpe::kCriticMaxOut) return fail(MPE_EUNSUPPORTED, "critic_create: out_dim out of range");
  DeviceGuard g(cfg->device);
  if (!g.ok) return fail(MPE_ECUDA, "critic_create: cannot select device");
  MpeCritic *c = new (std::nothrow) MpeCritic();
  if (c == nullptr) return fail(MPE_EINVAL, "critic_create: out of host memory");
  c->device = cfg->device;
  mpe::critic_layout(cfg->obs_dim, cfg->act_dim, cfg->out_dim, cfg->has_reward_head != 0, cfg->relu_attention != 0, &c->dev);
  cudaError_t e = cudaMalloc(&c->dev.blob, c->dev.blob_floats * sizeof(float));
  if (e == cudaSuccess) e = cudaMemset(c->dev.blob, 0, c->dev.blob_floats * sizeof(float));
  size_t n[kCriticFields];
  critic_counts(c->dev, n);
  if (e == cudaSuccess) e = cudaMalloc(&c->stage, total(n) * sizeof(float));
  if (e != cudaSuccess) {
    critic_destroy(c);
    return fail_cuda(e, "critic_create: cudaMalloc");
  }
  *out = c;
  return MPE_OK;
}

int critic_destroy(MpeCritic *c) {
  if (c == nullptr) return MPE_OK;
  DeviceGuard g(c->device);
  cudaDeviceSynchronize();
  if (c->dev.blob != nullptr) cudaFree(c->dev.blob);
  if (c->stage != nullptr) cudaFree(c->stage);
  delete c;
  return MPE_OK;
}

static int check_critic_weights(const MpeCritic *c, const CriticWeights *w, const char *who) {
  const std::string n(who);
  if (c == nullptr || w == nullptr) return fail(MPE_EINVAL, n + ": null argument");
  if (!w->dense1_w || !w->dense1_b || !w->w_ih || !w->w_hh || !w->b_ih || !w->b_hh || !w->dense2_w || !w->dense2_b)
    return fail(MPE_EINVAL, n + ": missing tensor");
  if (c->dev.has_r && (!w->dense3_w || !w->dense3_b)) return fail(MPE_EINVAL, n + ": missing dense3");
  return MPE_OK;
}

// Same scheme as actor_load: staged copy of the host tensors, the pack kernel, one synchronise.
int critic_load(MpeCritic *c, const CriticWeights *w, void *stream) {
  if (int rc = check_critic_weights(c, w, "critic_load")) return rc;
  DeviceGuard g(c->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  size_t n[kCriticFields];
  critic_counts(c->dev, n);
  CriticWeights staged = {};
  float *p = c->stage;
  for (int f = 0; f < kCriticFields; ++f) {
    if (n[f] == 0) continue;
    CK(cudaMemcpyAsync(p, w->*kCriticField[f], n[f] * sizeof(float), cudaMemcpyHostToDevice, st));
    staged.*kCriticField[f] = p;
    p += n[f];
  }
  CK(mpe::launch_critic_pack(c->dev, staged, st));
  CK(cudaStreamSynchronize(st));
  return MPE_OK;
}

int critic_load_device(MpeCritic *c, const CriticWeights *w, void *stream) {
  if (int rc = check_critic_weights(c, w, "critic_load_device")) return rc;
  size_t n[kCriticFields];
  critic_counts(c->dev, n);
  CriticWeights src = {};
  for (int f = 0; f < kCriticFields; ++f) {
    if (n[f] == 0) continue;
    if (!device_memory(w->*kCriticField[f], c->device))
      return fail(MPE_EINVAL, "critic_load_device: a weight pointer is not device memory on the critic's device");
    src.*kCriticField[f] = w->*kCriticField[f];
  }
  DeviceGuard g(c->device);
  CK(mpe::launch_critic_pack(c->dev, src, static_cast<cudaStream_t>(stream)));
  return MPE_OK;
}

int critic_forward(MpeCritic *c, const float *obs, const float *action, int64_t B, int32_t N, float *q, float *r,
                   void *stream) {
  if (c == nullptr || obs == nullptr || action == nullptr || q == nullptr) return fail(MPE_EINVAL, "critic_forward: null argument");
  if (B <= 0) return MPE_OK;
  if (N < 1 || N > mpe::kCriticMaxAgents) return fail(MPE_EUNSUPPORTED, "critic_forward: 1..16 agents");
  if (r != nullptr && !c->dev.has_r) return fail(MPE_EINVAL, "critic_forward: no reward head loaded");
  DeviceGuard g(c->device);
  CK(mpe::launch_critic_forward(c->dev, obs, action, B, N, q, r, static_cast<cudaStream_t>(stream)));
  return MPE_OK;
}

int64_t critic_backward_workspace(MpeCritic *c, int64_t B, int32_t N) {
  if (c == nullptr) return fail(MPE_EINVAL, "critic_backward_workspace: null critic");
  if (B < 0) return fail(MPE_EINVAL, "critic_backward_workspace: B < 0");
  if (N < 1 || N > mpe::kCriticMaxAgents) return fail(MPE_EUNSUPPORTED, "critic_backward_workspace: 1..16 agents");
  return mpe::critic_backward_bytes(c->dev, B, N);
}

int critic_backward(MpeCritic *c, const float *obs, const float *action, int64_t B, int32_t N, const float *dq,
                    const float *dr, float *dobs, float *daction, const CriticGrads *grads, void *workspace,
                    int64_t workspace_bytes, void *stream) {
  if (c == nullptr || obs == nullptr || action == nullptr || dq == nullptr || workspace == nullptr)
    return fail(MPE_EINVAL, "critic_backward: null argument");
  if (B < 0) return fail(MPE_EINVAL, "critic_backward: B < 0");
  if (N < 1 || N > mpe::kCriticMaxAgents) return fail(MPE_EUNSUPPORTED, "critic_backward: 1..16 agents");
  const CriticGrads none = {};
  const CriticGrads &g = grads != nullptr ? *grads : none;
  if (!c->dev.has_r && (dr != nullptr || g.dense3_w != nullptr || g.dense3_b != nullptr))
    return fail(MPE_EINVAL, "critic_backward: dr / dense3 gradients on a critic without a reward head");
  const int64_t need = mpe::critic_backward_bytes(c->dev, B, N);
  if (workspace_bytes < need)
    return fail(MPE_EINVAL, "critic_backward: workspace of " + std::to_string(workspace_bytes) + " bytes, " +
                                std::to_string(need) + " needed");
  if (B == 0) return MPE_OK;
  const void *ptrs[] = {obs, action, dq, dr, dobs, daction, workspace, g.dense1_w, g.dense1_b, g.w_ih, g.w_hh,
                        g.b_ih, g.b_hh, g.dense2_w, g.dense2_b, g.dense3_w, g.dense3_b};
  for (const void *p : ptrs)
    if (p != nullptr && !device_memory(p, c->device))
      return fail(MPE_EINVAL, "critic_backward: a pointer is not device memory on the critic's device");
  DeviceGuard dg(c->device);
  CK(mpe::launch_critic_backward(c->dev, obs, action, B, N, dq, dr, dobs, daction, g, workspace,
                                 static_cast<cudaStream_t>(stream)));
  return MPE_OK;
}

// ------------------------------------------------------------------------------------------------
// replay ring
// ------------------------------------------------------------------------------------------------
int replay_create(const ReplayConfig *cfg, MpeReplay **out) {
  if (cfg == nullptr || out == nullptr) return fail(MPE_EINVAL, "replay_create: null argument");
  *out = nullptr;
  if (cfg->capacity <= 0 || cfg->num_agents <= 0 || cfg->num_agents > 32 || cfg->obs_dim <= 0 || cfg->act0 <= 0 ||
      cfg->act0 > 127 || cfg->act1 < 0 || cfg->act1 > 127)
    return fail(MPE_EINVAL, "replay_create: bad configuration");
  const int64_t rec = mpe::ReplayDev::record_bytes(cfg->num_agents, cfg->obs_dim);
  if (rec > mpe::kReplayMaxRecordBytes)  // replay_add could never fill such a ring
    return fail(MPE_EUNSUPPORTED, "replay_create: a transition record of " + std::to_string(rec) +
                                      " bytes exceeds the " + std::to_string(mpe::kReplayMaxRecordBytes) + "-byte limit");
  DeviceGuard g(cfg->device);
  if (!g.ok) return fail(MPE_ECUDA, "replay_create: cannot select device");
  MpeReplay *r = new (std::nothrow) MpeReplay();
  if (r == nullptr) return fail(MPE_EINVAL, "replay_create: out of host memory");
  r->device = cfg->device;
  mpe::ReplayDev &d = r->dev;
  d.capacity = cfg->capacity; d.N = cfg->num_agents; d.D = cfg->obs_dim; d.A0 = cfg->act0; d.A1 = cfg->act1;
  d.rec_bytes = rec;
  cudaError_t e = cudaMalloc(&d.ring, (size_t)d.capacity * (size_t)d.rec_bytes);
  if (e != cudaSuccess) {
    replay_destroy(r);
    return fail_cuda(e, "replay_create: cudaMalloc");
  }
  *out = r;
  return MPE_OK;
}

int replay_destroy(MpeReplay *r) {
  if (r == nullptr) return MPE_OK;
  DeviceGuard g(r->device);
  cudaDeviceSynchronize();
  void *ptrs[] = {r->dev.ring, r->idx_scratch};
  for (void *p : ptrs)
    if (p != nullptr) cudaFree(p);
  delete r;
  return MPE_OK;
}

int replay_clear(MpeReplay *r) {
  if (r == nullptr) return fail(MPE_EINVAL, "replay_clear: null handle");
  r->size = 0; r->head = 0;
  return MPE_OK;
}

int64_t replay_len(const MpeReplay *r) { return r == nullptr ? 0 : r->size; }
int64_t replay_next_idx(const MpeReplay *r) { return r == nullptr ? 0 : r->head; }

int replay_add(MpeReplay *r, const float *obs, const int32_t *act_u, const int32_t *act_c, const float *rew,
               const float *obs_next, const float *done, int64_t B, void *stream) {
  if (r == nullptr || obs == nullptr || act_u == nullptr || rew == nullptr || obs_next == nullptr)
    return fail(MPE_EINVAL, "replay_add: null argument");
  if (B <= 0) return MPE_OK;
  if (B > r->dev.capacity) return fail(MPE_EINVAL, "replay_add: batch larger than the ring");
  if (r->dev.A1 > 0 && act_c == nullptr) return fail(MPE_EINVAL, "replay_add: act_c required for a two-head actor");
  DeviceGuard g(r->device);
  CK(mpe::launch_replay_add(r->dev, r->head, B, obs, act_u, act_c, rew, obs_next, done, static_cast<cudaStream_t>(stream)));
  r->head = (r->head + B) % r->dev.capacity;
  r->size = r->size + B < r->dev.capacity ? r->size + B : r->dev.capacity;
  return MPE_OK;
}

int replay_sample(MpeReplay *r, int64_t batch, const int64_t *idx, uint64_t seed, float *obs, float *act_onehot,
                  float *rew, float *obs_next, float *done, int64_t *idx_out, void *stream) {
  if (r == nullptr) return fail(MPE_EINVAL, "replay_sample: null handle");
  if (batch <= 0) return MPE_OK;
  if (r->size <= 0) return fail(MPE_EINVAL, "replay_sample: the ring is empty");
  DeviceGuard g(r->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t *use = idx;
  if (idx == nullptr) {  // ReplayBuffer.make_index: uniform with replacement, into idx_out or a private scratch
    int64_t *dst = idx_out;
    if (dst == nullptr) {
      if (batch > r->idx_cap) {
        if (r->idx_scratch != nullptr) cudaFree(r->idx_scratch);
        r->idx_scratch = nullptr; r->idx_cap = 0;
        CK(cudaMalloc(&r->idx_scratch, (size_t)batch * sizeof(int64_t)));
        r->idx_cap = batch;
      }
      dst = r->idx_scratch;
    }
    CK(mpe::launch_replay_make_index(r->size, batch, seed, r->draws, dst, st));
    use = dst;
  } else if (idx_out != nullptr) {
    CK(cudaMemcpyAsync(idx_out, idx, (size_t)batch * sizeof(int64_t), cudaMemcpyDeviceToDevice, st));
  }
  if (obs != nullptr || act_onehot != nullptr || rew != nullptr || obs_next != nullptr || done != nullptr)
    CK(mpe::launch_replay_gather(r->dev, r->size, batch, use, obs, act_onehot, rew, obs_next, done, st));
  if (idx == nullptr) r->draws += 1;
  return MPE_OK;
}

}  // extern "C"

// precision dispatch for the env launchers declared in env_launch.h
namespace mpe {
bool env_supported(int scenario, int N) {
  if (scenario == 0) return N >= 1 && N <= 12;  // simple_spread: make_world(num_agents=n), experiments/scenarios.py:170
  if (scenario == 3) return N == 8;  // fullobs_collect_treasure
  return (scenario == 1 || scenario == 2) && N == 2;
}
cudaError_t launch_reset(const EnvStateAny &a, const uint8_t *mask, void *obs, int auto_len, cudaStream_t st) {
  return a.precision == MPE_F64 ? launch_reset_f64(a, mask, obs, auto_len, st) : launch_reset_f32(a, mask, obs, auto_len, st);
}
cudaError_t launch_observe(const EnvStateAny &a, void *obs, cudaStream_t st) {
  return a.precision == MPE_F64 ? launch_observe_f64(a, obs, st) : launch_observe_f32(a, obs, st);
}
cudaError_t launch_step(const EnvStateAny &a, const int32_t *act_u, const int32_t *act_c, const void *comm_vec,
                        void *obs, void *rew, uint8_t *done, int32_t *info_i, void *info_f, cudaStream_t st) {
  return a.precision == MPE_F64 ? launch_step_f64(a, act_u, act_c, comm_vec, obs, rew, done, info_i, info_f, st)
                                : launch_step_f32(a, act_u, act_c, comm_vec, obs, rew, done, info_i, info_f, st);
}
cudaError_t launch_set_state(const EnvStateAny &a, const void *pos, const void *vel, const void *lm,
                             const int32_t *goal, cudaStream_t st) {
  return a.precision == MPE_F64 ? launch_set_state_f64(a, pos, vel, lm, goal, st)
                                : launch_set_state_f32(a, pos, vel, lm, goal, st);
}
cudaError_t launch_get_state(const EnvStateAny &a, void *pos, void *vel, void *lm, int32_t *goal, cudaStream_t st) {
  return a.precision == MPE_F64 ? launch_get_state_f64(a, pos, vel, lm, goal, st)
                                : launch_get_state_f32(a, pos, vel, lm, goal, st);
}
}  // namespace mpe
