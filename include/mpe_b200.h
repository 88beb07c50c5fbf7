/*
 * mpe_b200.h - C ABI of libmpe_b200.so: batched multi-agent particle environment
 * step + observe + reward and the rls actor forward, hand-written for sm_100a.
 *
 * Every entry point below replaces a piece of the Python hot path of
 * yjpark1/multiagent_rl (paths relative to the reference tree).  The physics
 * lives in the third-party `multiagent` package the reference imports at
 * experiments/scenarios.py:2-3; for those rows the reference CALL SITE is cited.
 *
 * Conventions
 *   - plain C: opaque handles, PODs, raw pointers; no C++/torch types.
 *   - return 0 on success, <0 on failure (MPE_E*); text via mpe_last_error()
 *     (thread-local).  Nothing throws, nothing exits.
 *   - all pointers are DEVICE pointers unless the name ends in `_host`.
 *   - buffers are borrowed: the caller allocates and keeps them alive until the
 *     work enqueued on `stream` (a cudaStream_t passed as void*) has finished.
 *     Handles own only their persistent state and free it in *_destroy.
 *   - nothing synchronises the host except the *_host entry points, *_destroy,
 *     mpe_stats_read, actor_load and critic_load.
 *   - a handle is not thread-safe; handles on different devices are independent.
 *     One MpeActor may serve several MpeEnv handles on DIFFERENT streams at the same time through mpe_rollout and
 *     mpe_act_step_host_async (scratch per env handle); actor_forward and actor_forward_host calls on one actor must
 *     stay on one stream at a time (teams of > 3 agents and two-head actors park partial logits in the actor's own
 *     scratch buffer).
 *   - "real" is float for MPE_F32 handles and double for MPE_F64 (validation build).
 *   - tensor layouts are row-major with the env index outermost: obs[B][N][D],
 *     rew[B][N], done[B][N], act[B][N].
 */
#ifndef MPE_B200_H_
#define MPE_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MPE_ABI_VERSION 9

enum { MPE_OK = 0, MPE_EINVAL = -1, MPE_ECUDA = -2, MPE_EUNSUPPORTED = -3 };
enum { MPE_SIMPLE_SPREAD = 0, MPE_SIMPLE_REFERENCE = 1, MPE_SIMPLE_SPEAKER_LISTENER = 2,
       MPE_COLLECT_TREASURE = 3 /* fullobs_collect_treasure, main.py:24-25; 6 collectors + 2 deposits, 6 treasures */ };
enum { MPE_F32 = 0, MPE_F64 = 1 };

typedef struct MpeEnv MpeEnv;     /* one shard of env instances on one GPU */
typedef struct MpeActor MpeActor; /* actor weights resident on one GPU */

/* What experiments/scenarios.py:124-192 (make_env) + Scenario.make_world fix. */
typedef struct {
  int32_t scenario;        /* MPE_SIMPLE_*                                            */
  int32_t num_agents;      /* 0 = scenario default; simple_spread: N = L (scenarios.py:170) */
  int32_t precision;       /* MPE_F32 | MPE_F64                                       */
  int32_t device;          /* CUDA ordinal                                            */
  int64_t num_envs;        /* B: env instances in this shard                          */
  int64_t env_id_offset;   /* global id of env 0 (multi-GPU sharding; keys the RNG)   */
  uint64_t seed;           /* Philox key (main.py:41-45 seed)                         */
  int32_t max_episode_len; /* rls/arglist.py:5 (25); used by mpe_rollout auto-reset   */
  int32_t reserved0;
  double max_speed;        /* Entity.max_speed; < 0 = None                            */
  double accel;            /* Entity.accel;     < 0 = None (sensitivity 5.0)          */
} MpeConfig;

typedef struct {
  int32_t num_agents, num_landmarks, obs_dim, dim_c;
  int32_t act_u;           /* width of the movement head (5)                          */
  int32_t act_c;           /* width of the message head (0 = no second head)          */
  int32_t precision, device;
  int64_t num_envs, env_id_offset;
} MpeDims;

int mpe_abi_version(void);
const char *mpe_last_error(void);

/* MultiAgentEnv(...) construction - experiments/scenarios.py:150-191 */
int mpe_create(const MpeConfig *cfg, MpeEnv **out);
int mpe_destroy(MpeEnv *env);
int mpe_query(const MpeEnv *env, MpeDims *out);
/* env.seed(seed) - main.py:45.  Enqueued on `stream`: new Philox key, episode indices restart at 0 with the next
 * reset, per-episode step counters and running returns are cleared. */
int mpe_seed(MpeEnv *env, uint64_t seed, void *stream);

/* env.reset() - experiments/run.py:28,60 -> upstream Scenario.reset_world + observation.
 * mask[B] (uint8, may be NULL = all) selects which envs start a new episode; positions ~ U[-1,1)^2,
 * velocities 0, goals uniform, drawn from Philox4x32-10 keyed by (seed, global env id, episode
 * index).  obs_out [B][N][D] may be NULL. */
int mpe_reset(MpeEnv *env, const uint8_t *mask, void *obs_out, void *stream);

/* State injection / readback (parity tests; host-drawn resets that mirror upstream's
 * np.random order).  pos/vel [B][N][2] real, lm [B][L][2] real, goal [B][N] int32 (-1 = None);
 * any pointer may be NULL to skip it.  MPE_COLLECT_TREASURE: lm = the six treasure positions and goal[b][0] = the
 * env's state word (bit l: type of treasure l; bit 6 + l: alive; bits 12 + 2 i: what collector i holds, 0 = nothing,
 * 1 + type otherwise); goal[b][1..] is ignored / left at -1. */
int mpe_set_state(MpeEnv *env, const void *pos, const void *vel, const void *lm, const int32_t *goal,
                  void *stream);
int mpe_get_state(MpeEnv *env, void *pos, void *vel, void *lm, int32_t *goal, void *stream);

/* scenario.observation(agent, world) for every agent - experiments/scenarios.py:6-63 */
int mpe_observe(MpeEnv *env, void *obs_out, void *stream);

/* env.step(action_n) - experiments/run.py:44 -> upstream MultiAgentEnv.step:
 *   _set_action (argmax -> one-hot -> u = (a1-a2, a3-a4) * 5.0), World.step
 *   (apply_action_force, apply_environment_force/get_collision_force, integrate_state,
 *   update_agent_state), then per agent observation (scenarios.py:6-63) and Scenario.reward.
 * act_u [B][N] int32 in 0..4 (the argmax index of the movement head);
 * act_c [B][N] int32 message index, or comm_vec [B][N][dim_c] real message (either may be NULL;
 *   only read for scenarios with a talking agent);
 * obs [B][N][D] real, rew [B][N] real, done [B][N] uint8 (always 0: no done_callback,
 *   scenarios.py:186-190), info_i [B][N+1] int32 = benchmark_data collisions per agent +
 *   occupied landmarks, info_f [B] real = benchmark_data min_dists; each output may be NULL.
 * MPE_COLLECT_TREASURE (experiments/scenarios.py:95-121,174-190 + the MAAC fork's scenario): sensitivity = accel,
 *   mass-aware contact forces, max_speed clip; observation / reward are taken BEFORE Scenario.post_step (pick-up,
 *   respawn, deposit), which runs at the end of the same kernel; info_i [B][N+1] = benchmark_data per agent (0 / 1)
 *   and a zero; info_f is not written.  The per-env episode step counter advances whether or not returns are tracked
 *   (it keys the respawn draws). */
int mpe_step(MpeEnv *env, const int32_t *act_u, const int32_t *act_c, const void *comm_vec, void *obs,
             void *rew, uint8_t *done, int32_t *info_i, void *info_f, void *stream);

/* Same call with HOST buffers (pinned or pageable): H2D of the actions, the step, D2H of
 * obs/rew/done, then a stream synchronise.  This is what a list-of-numpy caller pays. */
int mpe_step_host(MpeEnv *env, const int32_t *act_u_host, const int32_t *act_c_host, void *obs_host,
                  void *rew_host, uint8_t *done_host, void *stream);
/* env.reset() (experiments/run.py:28,60) + D2H of the observations, ENQUEUED on `stream` without a synchronise.
 * obs_host must be pinned and stay untouched until mpe_host_wait(stream). */
int mpe_reset_host_async(MpeEnv *env, void *obs_host, void *stream);
/* cudaStreamSynchronize(stream): everything the *_host_async calls enqueued on it has landed in host memory. */
int mpe_host_wait(void *stream);
/* One iteration of experiments/run.py:36-44 for a caller whose observations live in host memory:
 *   get_exploration_action(obs) -> env.step(action)
 * as H2D obs_host [B][N][D] -> actor forward + sample (Philox keyed by the env's seed, global env ids and `step`) ->
 * env step on the sampled actions -> ONE D2H of the transition block {act_u, act_c, obs', rew, done} laid out as
 * mpe_host_block_layout says (offsets in bytes, each 256 B aligned; act_u / act_c int32 [B][N], obs' fp32 [B][N][D],
 * rew fp32 [B][N], done uint8 [B][N]; act_c has zero length - off_act_c == off_obs - for envs without a message head).
 * Compared with the blocking actor_forward_host + mpe_step_host pair the sampled actions are not bounced through the
 * host before the step reads them and the four downloads are one copy; every step still uploads the observations and
 * downloads everything the two calls return.  Enqueued on `stream`, no host synchronisation (mpe_host_wait).
 * fp32 envs. */
typedef struct {
  uint64_t off_act_u, off_act_c, off_obs, off_rew, off_done, bytes;
} MpeHostBlockLayout;
int mpe_host_block_layout(const MpeEnv *env, MpeHostBlockLayout *out);
int mpe_act_step_host_async(MpeEnv *env, MpeActor *actor, const float *obs_host, uint64_t step, void *block_host,
                            void *stream);
/* Page-locked staging memory for the *_host entry points, straight from cudaHostAlloc.  (Measured on the B200 pool:
 * uploads from cudaHostAlloc memory run at 54 GB/s, from torch's pin_memory() blocks at 14 - 18 GB/s - torch 2.11's
 * caching host allocator hands out memory the copy engine reads three times slower; tools/h2d_probe.py.) */
int mpe_host_alloc(void **out, uint64_t bytes);
int mpe_host_free(void *p);

/* Episode-return bookkeeping (experiments/run.py:23-24,55-57,86-88).  When enabled, every mpe_step adds
 * sum_n rew to a per-env accumulator; mpe_reset folds finished episodes into
 * stats = {sum(ret), sum(ret^2), n_episodes, n_steps, n_nonfinite_episodes}.  Upstream's collision force divides by
 * the pair distance without an epsilon, so coincident agents produce NaN (reproduced, not masked): an episode whose
 * return is not finite is counted in stats[4] and left out of the two sums.
 * mpe_rollout ALWAYS keeps these counters (its auto-reset needs the per-env episode step) and folds every episode
 * it finishes, whatever mpe_track_returns says. */
#define MPE_STATS_LEN 5
int mpe_track_returns(MpeEnv *env, int32_t enable);
int mpe_stats_read(MpeEnv *env, double out[MPE_STATS_LEN], int32_t clear, void *stream); /* host sync */
int mpe_stats_ptr(MpeEnv *env, double **dev_ptr); /* device pointer to the MPE_STATS_LEN doubles (for NCCL) */

/* ---- actor: rls/model/ac_network_multi_gumbel.py:24-67 (+ ac_network_model_multi_gumbel.py) ---- */
typedef struct {
  int32_t obs_dim;   /* D                                                           */
  int32_t act0;      /* width of dense2 / dense2_1                                  */
  int32_t act1;      /* width of dense2_2, 0 for a single head (out_dim not a list) */
  int32_t has_model_head; /* dense3: 64 -> D (ac_network_model_multi_gumbel.py:49)  */
  int32_t device;
  int32_t reserved0;
} ActorConfig;

/* Pointers to fp32 tensors in the reference's state_dict layout (row-major [out][in], contiguous, 4 B alignment
 * suffices): HOST pointers for actor_load, DEVICE pointers for actor_load_device. */
typedef struct {
  const float *dense1_w, *dense1_b;               /* [64][D], [64]    */
  const float *w_ih, *w_hh, *b_ih, *b_hh;         /* [128][64], [128][32], [128], [128] */
  const float *w_ih_r, *w_hh_r, *b_ih_r, *b_hh_r; /* *_reverse        */
  const float *dense2_w, *dense2_b;               /* [act0][64], [act0]  (dense2 or dense2_1) */
  const float *dense2b_w, *dense2b_b;             /* [act1][64], [act1]  (dense2_2) or NULL   */
  const float *dense3_w, *dense3_b;               /* [D][64], [D] or NULL                     */
} ActorWeights;

int actor_create(const ActorConfig *cfg, MpeActor **out);
int actor_destroy(MpeActor *actor);
/* actor.load_state_dict(...) - rls/agent/multiagent/ddpg_gumbel_fix.py:231-241 - from HOST arrays: copies them to
 * the device, packs the weight images on `stream` and synchronises it; the arrays may be reused when it returns. */
int actor_load(MpeActor *actor, const ActorWeights *w, void *stream);
/* The same load from DEVICE tensors (a learner's parameters), enqueued on `stream` as one pack kernel: no host
 * synchronisation and no allocation, so it can be captured in a CUDA graph.  The tensors are read when the kernel
 * runs, not when the call returns: they must stay allocated until then, and a change made to them earlier on `stream`
 * is what gets loaded.  Ordering: actor launches on `stream` after this call see the new weights, launches enqueued
 * before it the old ones.  The weights are overwritten in place, so launches on OTHER streams (HostRollout shards
 * sharing this actor, for example) must be ordered against the load by the caller with events.  MPE_EINVAL before
 * anything is launched for a missing tensor (the rules of actor_load) or a pointer that is not device or managed
 * memory on the actor's device. */
int actor_load_device(MpeActor *actor, const ActorWeights *w, void *stream);

/* Implementation of the actor GEMMs: 0 = auto (tensor cores where supported), 1 = fp32 SIMT (FFMA),
 * 2 = tcgen05 tensor cores with fp16 hi/lo split operands (fp32-level accuracy; 2/3/4/6/8/9/12 agents).
 * Other values: MPE_EINVAL. */
int actor_set_impl(MpeActor *actor, int32_t impl);

/* Trainer.get_exploration_action - rls/agent/multiagent/ddpg_gumbel_fix.py:86-107:
 *   actor.forward (relu(dense1) -> BiLSTM over the agent axis -> relu -> dense2[_1,_2]) and
 *   F.gumbel_softmax(hard=True) == argmax(logits + G).
 * obs [B][N][D] fp32.  gumbel [B][N][act0+act1] fp32 injects the noise (parity mode); NULL draws it
 * from Philox keyed by (seed, env_id_offset + b, step, agent).  Outputs (each may be NULL):
 * logits [B][N][act0+act1], next_state [B][N][D] (model head), act_u [B][N] int32 (head 0 index),
 * act_c [B][N] int32 (head 1 index), onehot [B][N][act0+act1] fp32 (what the reference returns). */
int actor_forward(MpeActor *actor, const float *obs, int64_t B, int32_t N, const float *gumbel,
                  uint64_t seed, uint64_t step, int64_t env_id_offset, float *logits, float *next_state,
                  int32_t *act_u, int32_t *act_c, float *onehot, void *stream);
/* Same with HOST buffers: H2D obs, forward, D2H onehot / act, stream synchronise
 * (ddpg_gumbel_fix.py:93-94 and :100 are exactly these two copies). */
int actor_forward_host(MpeActor *actor, const float *obs_host, int64_t B, int32_t N, uint64_t seed,
                       uint64_t step, int64_t env_id_offset, int32_t *act_u_host, int32_t *act_c_host,
                       float *onehot_host, void *stream);

/* Gradients of the actor forward for Trainer.optimize() (ddpg_gumbel_fix.py:131-219): the actor loss through the
 * weights.  Output tensors are fp32 in the reference's state_dict layout ([out][in]), mirroring ActorWeights; a NULL
 * field is not computed.  bias_ih* and bias_hh* of a direction get the same gradient. */
typedef struct {
  float *dense1_w, *dense1_b;               /* [64][D], [64]    */
  float *w_ih, *w_hh, *b_ih, *b_hh;         /* [128][64], [128][32], [128], [128] */
  float *w_ih_r, *w_hh_r, *b_ih_r, *b_hh_r; /* *_reverse        */
  float *dense2_w, *dense2_b;               /* [act0][64], [act0]  (dense2 or dense2_1) */
  float *dense2b_w, *dense2b_b;             /* [act1][64], [act1]  (dense2_2); two-head actors only */
  float *dense3_w, *dense3_b;               /* [D][64], [D]; "+model" actors only       */
} ActorGrads;
/* Bytes of device workspace actor_backward needs for B samples of N agents (0 for B = 0); < 0 (MPE_E*) on error. */
int64_t actor_backward_workspace(MpeActor *actor, int64_t B, int32_t N);
/* Backward of the fp32 FFMA actor forward (actor_set_impl 1) on obs [B][N][D], with the weights of the last
 * actor_load* enqueued on `stream` (the forward is recomputed; nothing is kept from an earlier actor_forward).
 * dlogits [B][N][act0+act1] is the gradient of the loss with respect to the logits (both heads concatenated);
 * dnext_state [B][N][D] that with respect to next_state, for the "+model" actor only, NULL meaning zero.  Outputs,
 * each optional (NULL: not computed) and overwritten, never accumulated: dobs [B][N][D] and the fields of `grads`
 * (which may itself be NULL).  `workspace` is device memory of at least actor_backward_workspace(actor, B, N) bytes,
 * borrowed like every buffer; calls on different streams need different workspaces.  Enqueued on `stream`: no host
 * synchronisation, no allocation.  Deterministic: no floating-point atomics, every sum in an order that depends on B
 * and N alone, and a sample's dobs does not depend on where it sits in the batch.  MPE_EINVAL before any launch for a
 * null actor / obs / dlogits / workspace, dnext_state or dense3 gradients on an actor without a model head, dense2b
 * gradients on a single-head actor, a workspace that is too small, B < 0, or a pointer that is not device memory on
 * the actor's device; MPE_EUNSUPPORTED for N outside 1..12. */
int actor_backward(MpeActor *actor, const float *obs, int64_t B, int32_t N, const float *dlogits,
                   const float *dnext_state, float *dobs, const ActorGrads *grads, void *workspace,
                   int64_t workspace_bytes, void *stream);

/* The loop body of experiments/run.py:36-65 fused: for t in [0, T): observe -> actor -> sample ->
 * step -> reward -> (episode_step == max_episode_len ? reset), state never leaving the SM between
 * the actor and the physics.  F32 envs only.  Per-step outputs (each may be NULL) are written
 * at [t][...]: obs_next [T][B][N][D], rew [T][B][N], act_u [T][B][N], act_c [T][B][N],
 * info_i [T][B][N+1] int32 and info_f [T][B] fp32: benchmark_data, at [t] bit for bit what mpe_step writes to its
 * info_i / info_f for that step (collisions per agent + occupied landmarks, and min_dists; for
 * MPE_COLLECT_TREASURE the 0 / 1 flags per agent + a zero, and info_f is not written).  A NULL output changes
 * nothing else the call writes.
 * `step0` is the global step index of t = 0 (keys the Gumbel stream). */
int mpe_rollout(MpeEnv *env, MpeActor *actor, int32_t T, uint64_t step0, float *obs_next, float *rew,
                int32_t *act_u, int32_t *act_c, int32_t *info_i, void *info_f, void *stream);

/* ---- critic: rls/model/ac_network_multi_gumbel.py:70-148 (main.py path) and
 * rls/model/ac_network_model_multi_gumbel.py:69-143 ("+model": extra reward head, no relu after the attention).
 * Not on the acting path (SURVEY 8f-2): evaluated by Trainer.optimize() at ddpg_gumbel_fix.py:151,159,191. ---- */
typedef struct MpeCritic MpeCritic;
typedef struct {
  int32_t obs_dim;          /* D                                                           */
  int32_t act_dim;          /* sum of the action head widths (input = D + act_dim, main.py:61) */
  int32_t out_dim;          /* 1                                                           */
  int32_t has_reward_head;  /* dense3 (ac_network_model_multi_gumbel.py:91,141)            */
  int32_t relu_attention;   /* 1: relu on the attention output (ac_network_multi_gumbel.py:141), 0: "+model" critic */
  int32_t device;
} CriticConfig;
/* Pointers to fp32 tensors in the reference's state_dict layout (row-major [out][in], contiguous, 4 B alignment
 * suffices): HOST pointers for critic_load, DEVICE pointers for critic_load_device. */
typedef struct {
  const float *dense1_w, *dense1_b;        /* [64][D + act_dim], [64]                    */
  const float *w_ih, *w_hh, *b_ih, *b_hh;  /* lstm.*_l0: [256][64], [256][64], [256], [256] */
  const float *dense2_w, *dense2_b;        /* [out_dim][64], [out_dim]                   */
  const float *dense3_w, *dense3_b;        /* [out_dim][64], [out_dim] or NULL           */
} CriticWeights;
int critic_create(const CriticConfig *cfg, MpeCritic **out);
int critic_destroy(MpeCritic *critic);
/* From HOST arrays, like actor_load: copy, pack on `stream`, synchronise. */
int critic_load(MpeCritic *critic, const CriticWeights *w, void *stream);
/* From DEVICE tensors, like actor_load_device: one pack kernel on `stream`, no host synchronisation, no allocation;
 * critic launches on `stream` after the call see the new weights, launches on other streams are ordered by the caller.
 * MPE_EINVAL before any launch for a missing tensor or a pointer that is not device memory on the critic's device. */
int critic_load_device(MpeCritic *critic, const CriticWeights *w, void *stream);
/* critic.forward(obs, action): obs [B][N][D], action [B][N][act_dim] fp32 (one-hot or soft; two heads concatenated
 * like ac_network_multi_gumbel.py:131-132) -> q [B][out_dim] and, for the "+model" critic, r [B][out_dim] (or NULL). */
int critic_forward(MpeCritic *critic, const float *obs, const float *action, int64_t B, int32_t N, float *q, float *r,
                   void *stream);
/* Gradients of critic.forward for Trainer.optimize() (ddpg_gumbel_fix.py:131-219): the TD loss through the weights,
 * the actor loss through the action.  Output tensors are fp32 in the reference's state_dict layout ([out][in]); a
 * NULL field is not computed.  lstm.bias_ih_l0 and lstm.bias_hh_l0 get the same gradient. */
typedef struct {
  float *dense1_w, *dense1_b;        /* [64][D + act_dim], [64]                    */
  float *w_ih, *w_hh, *b_ih, *b_hh;  /* lstm.*_l0: [256][64], [256][64], [256], [256] */
  float *dense2_w, *dense2_b;        /* [out_dim][64], [out_dim]                   */
  float *dense3_w, *dense3_b;        /* [out_dim][64], [out_dim]; reward head only */
} CriticGrads;
/* Bytes of device workspace critic_backward needs for B samples of N agents (0 for B = 0); < 0 (MPE_E*) on error. */
int64_t critic_backward_workspace(MpeCritic *critic, int64_t B, int32_t N);
/* Backward of critic_forward on the same obs [B][N][D] and action [B][N][act_dim], with the weights of the last
 * critic_load* enqueued on `stream` (the forward is recomputed; nothing is kept from an earlier critic_forward).
 * dq [B][out_dim] is the gradient of the loss with respect to q; dr [B][out_dim] that with respect to r, for the
 * "+model" critic only, NULL meaning zero.  Outputs, each optional (NULL: not computed) and overwritten, never
 * accumulated: dobs [B][N][D], daction [B][N][act_dim] and the fields of `grads` (which may itself be NULL).
 * `workspace` is device memory of at least critic_backward_workspace(critic, B, N) bytes, borrowed like every buffer;
 * calls on different streams need different workspaces.  Enqueued on `stream`: no host synchronisation, no
 * allocation.  Deterministic: no floating-point atomics, every sum in an order that depends on B and N alone, and a
 * sample's dobs / daction do not depend on where it sits in the batch.  MPE_EINVAL before any launch for a null
 * critic / obs / action / dq / workspace, dr or dense3 gradients on a critic without a reward head, a workspace that is
 * too small, B < 0, or a pointer that is not device memory on the critic's device; MPE_EUNSUPPORTED for N outside
 * 1..16. */
int critic_backward(MpeCritic *critic, const float *obs, const float *action, int64_t B, int32_t N, const float *dq,
                    const float *dr, float *dobs, float *daction, const CriticGrads *grads, void *workspace,
                    int64_t workspace_bytes, void *stream);

/* ---- device-resident replay ring: rls/replay_buffer.py:9-91 (ReplayBuffer), fed with the tuple of
 * experiments/run.py:46,52 (obs_n, action_n_env, rew_shared = sum(rew_n), new_obs_n, float(done)) ---- */
typedef struct MpeReplay MpeReplay;
typedef struct {
  int64_t capacity;    /* ReplayBuffer(size)                                   */
  int32_t num_agents, obs_dim;
  int32_t act0, act1;  /* head widths (one-hot actions are rebuilt on sample)  */
  int32_t device, reserved0;
} ReplayConfig;

/* MPE_EUNSUPPORTED when one transition record (record_bytes in csrc/replay_launch.h) exceeds 48 KB. */
int replay_create(const ReplayConfig *cfg, MpeReplay **out);
int replay_destroy(MpeReplay *replay);
int replay_clear(MpeReplay *replay);               /* ReplayBuffer.clear  */
int64_t replay_len(const MpeReplay *replay);       /* len(buffer)         */
int64_t replay_next_idx(const MpeReplay *replay);  /* buffer._next_idx    */
/* ReplayBuffer.add for B env instances, appended in env order: obs / obs_next [B][N][D] fp32, act_u / act_c [B][N]
 * int32 head indices, rew [B][N] fp32 per-agent rewards (summed to the shared reward), done [B] fp32 or NULL (0). */
int replay_add(MpeReplay *replay, const float *obs, const int32_t *act_u, const int32_t *act_c, const float *rew,
               const float *obs_next, const float *done, int64_t B, void *stream);
/* ReplayBuffer.make_index + sample_index: idx [batch] int64 device indices, or NULL to draw them uniformly with
 * replacement (Philox domain 5, keyed by seed and the number of draws so far).  Caller-supplied indices follow Python list
 * indexing of ReplayBuffer._storage: negative values count from the end; values still outside [0, len) are clamped
 * into the ring (never read out of bounds) - validate host-side where an IndexError is wanted.  Outputs (each may be NULL): obs / obs_next
 * [batch][N][D], act_onehot [batch][N][act0+act1], rew [batch], done [batch], idx_out [batch]. */
int replay_sample(MpeReplay *replay, int64_t batch, const int64_t *idx, uint64_t seed, float *obs, float *act_onehot,
                  float *rew, float *obs_next, float *done, int64_t *idx_out, void *stream);

/* mpe_rollout that also appends every env-step's transition to `replay`: (obs_t, act_u, act_c, sum_n rew,
 * obs_{t+1}, done = 0), where obs_t is the observation the actor acted on (the post-reset observation at an episode's
 * first step) and obs_{t+1} the one the step returned (before any reset).  Step-major, then env order: the ring ends
 * up as after T replay_add calls of B transitions each, wrapping as often as T * B / capacity says.  Recordings,
 * env state, Philox streams, episode statistics and info_i / info_f are those of mpe_rollout; the recording pointers
 * may be NULL.
 * The ring must match the env and actor (num_agents, obs_dim, act0 / act1), sit on their device and hold at least
 * B transitions; otherwise MPE_EINVAL before anything is launched.  Envs whose episodes are aligned (after an
 * unmasked reset) run the fused kernel in segments up to each episode end and one ring-writer launch per segment;
 * others run per-step kernels with one replay_add per step. */
int mpe_rollout_replay(MpeEnv *env, MpeActor *actor, MpeReplay *replay, int32_t T, uint64_t step0, float *obs_next,
                       float *rew, int32_t *act_u, int32_t *act_c, int32_t *info_i, void *info_f, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* MPE_B200_H_ */
