// Per-env device logic of the particle world: reset, discrete action -> force, pairwise soft-contact
// forces, damped integration, observation rows, rewards.  One thread owns one env and keeps every
// entity in registers (all loops below are fully unrolled over the compile-time agent count).
//
// Reference rows (paths relative to the reference tree; the physics is in the `multiagent` package
// imported at experiments/scenarios.py:2-3, so upstream function names are cited for those):
//   _set_action        MultiAgentEnv._set_action       (called from experiments/run.py:44)
//   physics()          World.step: apply_action_force, apply_environment_force /
//                      get_collision_force, integrate_state
//   obs_row()          experiments/scenarios.py:6-20, :23-42, :45-63
//   reward()           Scenario.reward / benchmark_data of simple_spread, simple_reference,
//                      simple_speaker_listener
// The arithmetic is written in the reference's operation order so that the fp64 instantiation
// (compiled with -fmad=false) differs from numpy only through exp/log1p rounding.
#pragma once
#include <cmath>
#include <type_traits>

#include "common.cuh"
#include "env_launch.h"

namespace mpe {

enum : int { kSpread = 0, kReference = 1, kSpeaker = 2, kTreasure = 3 };  // kTreasure: env_treasure.cuh

template <int SC, int N_>
struct Dims {
  static constexpr int N = N_;
  static constexpr int L = (SC == kSpread) ? N_ : 3;
  static constexpr int D = (SC == kSpread) ? 4 + 2 * L : (SC == kReference ? 21 : 11);
  static constexpr int DIMC = (SC == kSpread) ? 2 : (SC == kReference ? 10 : 3);
  static constexpr int R = N * D;  // obs floats per env
  static constexpr bool kCollide = (SC == kSpread);
  static constexpr bool kHasGoal = (SC != kSpread);
  static constexpr bool kTalks = (SC == kReference);  // comm visible in obs
};

// Device view of one shard's persistent state (structure-of-arrays over envs).
template <typename T>
struct EnvState {
  T *pv;              // [N][B][4]  {px, py, vx, vy}   (16 B vector per agent per env in fp32)
  T *lm;              // [L][B][2]  {x, y}
  int32_t *goal;      // [B]  goal landmark of agent0 | agent1 << 8   (0xFF = None)
  uint32_t *episode;  // [B]  episode index (Philox "t" of the reset stream)
  int32_t *tstep;     // [B]  steps taken in the current episode
  T *ep_ret;          // [B]  running episode return, summed over agents
  T *comm;            // [N][DIMC][B] last message of every agent (simple_reference only, else NULL)
  double *stats;      // [kStatsLen]  sum(ret), sum(ret^2), n_episodes, n_steps, n_nonfinite_episodes
  int64_t B;
  int64_t gid0;       // global id of env 0
  uint64_t seed;
  T max_speed;        // < 0: None
  T accel;            // < 0: None -> sensitivity 5.0
  int32_t track;      // accumulate episode returns
  // Exact squared-distance thresholds (set_thresholds): sqrt is monotone and correctly rounded, so
  //   sqrt(d2) < c  <=>  d2 < t2(c)      and      sqrt(d2) > c  <=>  d2 >= t2gt(c)
  // which lets the collision / occupancy flags and the far-pair early-out skip the square root bit-exactly.
  T t2_coll;          // sqrt(d2) < dist_min (0.30)          is_collision
  T t2_occ;           // sqrt(d2) < 0.1                      occupied landmark
  T t2_cut;           // sqrt(d2) > dist_min + underflow     contact force is exactly 0 beyond
  // fullobs_collect_treasure (env_treasure.cuh): contacts collector-collector / collector-deposit / collector-treasure,
  // force cut-offs collector-collector / collector-deposit / deposit-deposit
  T tr_t2[3], tr_cut[3];
};

// smallest x with sqrt(x) >= c  (so that  sqrt(d2) < c  <=>  d2 < x); host, IEEE sqrt
template <typename T>
inline T sqrt_lt_threshold(T c) {
  T x = c * c;
  while (std::sqrt(x) >= c) x = std::nextafter(x, (T)0);
  while (std::sqrt(x) < c) x = std::nextafter(x, (T)INFINITY);
  return x;
}
// smallest x with sqrt(x) > c  (so that  sqrt(d2) > c  <=>  d2 >= x)
template <typename T>
inline T sqrt_gt_threshold(T c) {
  T x = c * c;
  while (std::sqrt(x) > c) x = std::nextafter(x, (T)0);
  while (!(std::sqrt(x) > c)) x = std::nextafter(x, (T)INFINITY);
  return x;
}

template <typename T>
__device__ __forceinline__ T softplus_pen(T dist, T dist_min) {
  // np.logaddexp(0, -(dist - dist_min)/k) * k   with k = contact_margin
  const T k = (T)1e-3;
  const T y = -(dist - dist_min) / k;
  T r;
  if (y == (T)0) {
    r = (T)0.693147180559945309417232121458176568;
  } else {
    const T tmp = -y;
    if (tmp > (T)0)
      r = log1p(exp(-tmp));
    else if (tmp <= (T)0)
      r = y + log1p(exp(tmp));
    else
      r = tmp;  // NaN
  }
  return r * k;
}

template <typename T>
struct Underflow;  // (dist - dist_min) beyond which exp(-x/k) is exactly 0 in T, so the force is exactly 0
template <>
struct Underflow<float> {
  static constexpr float v = 0.105f;
};
template <>
struct Underflow<double> {
  static constexpr double v = 0.75;
};

// Fold finished episodes of a warp into stats = {sum ret, sum ret^2, episodes, steps, non-finite episodes}.
// Upstream divides by the pair distance without an epsilon, so coincident agents give NaN forces (replicated, not
// "fixed"); an episode whose return is not finite is COUNTED in stats[4] and kept out of the two sums, so one such
// episode does not poison the running statistics.  Mean return = stats[0] / (stats[2] - stats[4]).
__device__ __forceinline__ void fold_stats(double *stats, double ret, double n_ep, double n_steps) {
  if (!__any_sync(0xffffffffu, n_ep != 0.0)) return;  // no episode of this warp ended in this step (the usual case)
  const bool bad = n_ep != 0.0 && !(fabs(ret) <= 1.7976931348623157e308);
  double a = bad ? 0.0 : ret * n_ep, b = bad ? 0.0 : ret * ret * n_ep, c = n_ep, d = n_steps, e = bad ? 1.0 : 0.0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a += __shfl_xor_sync(0xffffffffu, a, o);
    b += __shfl_xor_sync(0xffffffffu, b, o);
    c += __shfl_xor_sync(0xffffffffu, c, o);
    d += __shfl_xor_sync(0xffffffffu, d, o);
    e += __shfl_xor_sync(0xffffffffu, e, o);
  }
  if ((threadIdx.x & 31) == 0 && c > 0.0) {
    atomicAdd(stats + 0, a);
    atomicAdd(stats + 1, b);
    atomicAdd(stats + 2, c);
    atomicAdd(stats + 3, d);
    if (e > 0.0) atomicAdd(stats + 4, e);
  }
}

template <typename T>
inline void set_thresholds(EnvState<T> &s, int scenario) {
  const T size = scenario == kSpread ? (T)0.15 : (scenario == kReference ? (T)0.05 : (T)0.075);
  const T dist_min = size + size;
  s.t2_coll = sqrt_lt_threshold<T>(dist_min);
  s.t2_occ = sqrt_lt_threshold<T>((T)0.1);
  s.t2_cut = sqrt_gt_threshold<T>(dist_min + Underflow<T>::v);
  for (int k = 0; k < 3; ++k) s.tr_t2[k] = s.tr_cut[k] = (T)0;
  if (scenario == kTreasure) {  // sizes: collector 0.05, deposit 0.075, treasure 0.025 (sums taken in double like numpy)
    const double cc = 0.05 + 0.05, cd = 0.05 + 0.075, ct = 0.05 + 0.025, dd = 0.075 + 0.075;
    s.tr_t2[0] = sqrt_lt_threshold<T>((T)cc);
    s.tr_t2[1] = sqrt_lt_threshold<T>((T)cd);
    s.tr_t2[2] = sqrt_lt_threshold<T>((T)ct);
    s.tr_cut[0] = sqrt_gt_threshold<T>((T)cc + Underflow<T>::v);
    s.tr_cut[1] = sqrt_gt_threshold<T>((T)cd + Underflow<T>::v);
    s.tr_cut[2] = sqrt_gt_threshold<T>((T)dd + Underflow<T>::v);
  }
}

// host side: the kernels' EnvState<T> view of a shard's type-erased EnvStateAny (env_launch.h)
template <typename T>
inline EnvState<T> typed(const EnvStateAny &a) {
  EnvState<T> s;
  s.pv = static_cast<T *>(a.pv);
  s.lm = static_cast<T *>(a.lm);
  s.goal = a.goal;
  s.episode = a.episode;
  s.tstep = a.tstep;
  s.ep_ret = static_cast<T *>(a.ep_ret);
  s.comm = static_cast<T *>(a.comm);
  s.stats = a.stats;
  s.B = a.B;
  s.gid0 = a.gid0;
  s.seed = a.seed;
  s.max_speed = (T)a.max_speed;
  s.accel = (T)a.accel;
  s.track = a.track;
  set_thresholds<T>(s, a.scenario);
  return s;
}

// get_collision_force for one close pair: (gx, gy) = contact_force * delta / dist * penetration.
// double: upstream's operation order (validation build).  float: same formula with the fast exp/log/reciprocal
// intrinsics - their error (<= 1e-6 relative on a force that is then scaled by dt = 0.1) is far inside the
// fp32-vs-float64 tolerance, and the pair is already known to be within reach of the softplus.
template <typename T>
__device__ __forceinline__ void contact_force(T dx, T dy, T d2, T dist_min, T &gx, T &gy) {
  if constexpr (std::is_same<T, float>::value) {
    // 3 MUFU ops (rsq, ex2, lg2) and ~12 FP32 ops, branch free: softplus(y) = max(y, 0) + log(1 + exp(-|y|)).
    // Far pairs give exp -> 0, log(1) = 0, i.e. exactly +-0 (the double build skips them with the same result);
    // coincident agents give NaN like upstream's 0/0.
    // raw MUFU forms: rsqrtf() / __expf() wrap the approx instructions in denormal-range handling (8 extra
    // instructions per pair) that cannot matter here - d2 is either 0 (coincident: inf -> NaN, as wanted) or far
    // above 2^-126, and exp results below 2^-126 vanish in the 1 + e that follows either way
    float rinv, e;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(rinv) : "f"(d2));
    const float dist = d2 * rinv;
    const float y = (dist_min - dist) * 1000.0f;  // -(dist - dist_min) / contact_margin
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(-fabsf(y) * 1.4426950408889634f));
    const float sp = fmaxf(y, 0.0f) + __logf(1.0f + e);
    const float sc = (0.1f * sp) * rinv;  // contact_force * (sp * contact_margin) / dist
    gx = __fmul_rn(dx, sc);  // never contracted into the caller's accumulation: every kernel variant
    gy = __fmul_rn(dy, sc);  // (thread-per-env, lanes-per-env, fused) produces the same bits
  } else {
    const T dist = sqrt(d2);
    const T pen = softplus_pen<T>(dist, dist_min);
    gx = (T)100 * dx / dist * pen;
    gy = (T)100 * dy / dist * pen;
  }
}

// a*a + b*b and a*b + c with a FIXED choice of which product is fused, so that every kernel variant (thread-
// per-env, lanes-per-env, fused rollout) rounds identically.  double (built with -fmad=false): numpy's order.
template <typename T>
__device__ __forceinline__ T sq2(T a, T b) { return a * a + b * b; }
template <>
__device__ __forceinline__ float sq2<float>(float a, float b) { return fmaf(a, a, __fmul_rn(b, b)); }
template <typename T>
__device__ __forceinline__ T mad(T a, T b, T c) { return a * b + c; }
template <>
__device__ __forceinline__ float mad<float>(float a, float b, float c) { return fmaf(a, b, c); }
template <typename T>
__device__ __forceinline__ T mul_rn(T a, T b) { return a * b; }
template <>
__device__ __forceinline__ float mul_rn<float>(float a, float b) { return __fmul_rn(a, b); }

// World.integrate_state for one movable entity (damping 0.25, mass 1, dt 0.1, optional max_speed clip)
template <typename T>
__device__ __forceinline__ void integrate_agent(T &px, T &py, T &vx, T &vy, T fx, T fy, T max_speed) {
  T vxi = mad<T>(fx, (T)0.1, mul_rn<T>(vx, (T)0.75));  // v = v * (1 - damping); v += (f / mass) * dt
  T vyi = mad<T>(fy, (T)0.1, mul_rn<T>(vy, (T)0.75));
  if (max_speed >= (T)0) {
    const T speed = sqrt(sq2<T>(vxi, vyi));
    if (speed > max_speed) {
      vxi = vxi / speed * max_speed;
      vyi = vyi / speed * max_speed;
    }
  }
  vx = vxi; vy = vyi;
  px = mad<T>(vxi, (T)0.1, px);
  py = mad<T>(vyi, (T)0.1, py);
}

template <typename T, int SC, int N>
struct Env {
  using Dm = Dims<SC, N>;
  static constexpr int L = Dm::L;
  static constexpr int D = Dm::D;
  T px[N], py[N], vx[N], vy[N];
  T lx[L], ly[L];
  int goal[2];  // landmark index or -1

  __device__ __forceinline__ static T size_of_agent() {
    return SC == kSpread ? (T)0.15 : (SC == kReference ? (T)0.05 : (T)0.075);
  }
  __device__ __forceinline__ static bool movable(int i) { return !(SC == kSpeaker && i == 0); }

  __device__ __forceinline__ void load(const EnvState<T> &s, int64_t b) {
#pragma unroll
    for (int i = 0; i < N; ++i) {
      const Vec4<T> v = ld4(s.pv + ((int64_t)i * s.B + b) * 4);
      px[i] = v.x; py[i] = v.y; vx[i] = v.z; vy[i] = v.w;
    }
#pragma unroll
    for (int l = 0; l < L; ++l) {
      const Vec2<T> v = ld2(s.lm + ((int64_t)l * s.B + b) * 2);
      lx[l] = v.x; ly[l] = v.y;
    }
    goal[0] = goal[1] = -1;
    if (Dm::kHasGoal) {
      const int32_t g = s.goal[b];
      goal[0] = (g & 0xFF) == 0xFF ? -1 : (g & 0xFF);
      goal[1] = ((g >> 8) & 0xFF) == 0xFF ? -1 : ((g >> 8) & 0xFF);
    }
  }

  __device__ __forceinline__ void store_agents(const EnvState<T> &s, int64_t b) const {
#pragma unroll
    for (int i = 0; i < N; ++i) st4(s.pv + ((int64_t)i * s.B + b) * 4, Vec4<T>{px[i], py[i], vx[i], vy[i]});
  }
  __device__ __forceinline__ void store_world(const EnvState<T> &s, int64_t b) const {
#pragma unroll
    for (int l = 0; l < L; ++l) st2(s.lm + ((int64_t)l * s.B + b) * 2, Vec2<T>{lx[l], ly[l]});
    if (Dm::kHasGoal) s.goal[b] = (goal[0] & 0xFF) | ((goal[1] & 0xFF) << 8);
  }

  // Scenario.reset_world: agents then landmarks ~ U[-1,1)^2, zero velocity, uniform goals.
  __device__ __forceinline__ void reset(uint64_t seed, uint64_t gid, uint32_t episode) {
    constexpr int E = N + L;
#pragma unroll
    for (int j = 0; j < (E + 1) / 2; ++j) {
      const uint4 r = philox_raw(seed, gid, episode, kDomainReset, j);
      set_entity_pos(2 * j, bits_to_pos<T>(r.x), bits_to_pos<T>(r.y));
      if (2 * j + 1 < E) set_entity_pos(2 * j + 1, bits_to_pos<T>(r.z), bits_to_pos<T>(r.w));
    }
#pragma unroll
    for (int i = 0; i < N; ++i) vx[i] = vy[i] = (T)0;
    goal[0] = goal[1] = -1;
    if (Dm::kHasGoal) {
      const uint4 r = philox_raw(seed, gid, episode, kDomainGoal, 0);
      goal[0] = (int)__umulhi(r.x, (uint32_t)L);
      if (SC == kReference) goal[1] = (int)__umulhi(r.y, (uint32_t)L);
    }
  }
  __device__ __forceinline__ void set_entity_pos(int e, T x, T y) {
    // e is a compile-time constant after unrolling
    if (e < N) { px[e] = x; py[e] = y; }
    else { lx[e - N] = x; ly[e - N] = y; }
  }

  // _set_action (one-hot branch) + World.step up to integrate_state.
  __device__ __forceinline__ void physics(const int *act_u, const EnvState<T> &s) {
    const T max_speed = s.max_speed;
    const T sens = s.accel >= (T)0 ? s.accel : (T)5.0;
    T fx[N], fy[N];
#pragma unroll
    for (int i = 0; i < N; ++i) {
      const int a = act_u[i];
      // u[0] += a[1] - a[2]; u[1] += a[3] - a[4]; u *= sensitivity
      const T u0 = (T)0 + ((a == 1 ? (T)1 : (T)0) - (a == 2 ? (T)1 : (T)0));
      const T u1 = (T)0 + ((a == 3 ? (T)1 : (T)0) - (a == 4 ? (T)1 : (T)0));
      fx[i] = u0 * sens;
      fy[i] = u1 * sens;
    }
    if (Dm::kCollide) {
      const T dist_min = size_of_agent() + size_of_agent();
#pragma unroll
      for (int a = 0; a < N; ++a) {
#pragma unroll
        for (int b = a + 1; b < N; ++b) {
          const T dx = px[a] - px[b], dy = py[a] - py[b];
          const T d2 = sq2<T>(dx, dy);
          // double: skip pairs whose penalty underflows to exactly 0; float: branch-free (adds an exact zero)
          if (std::is_same<T, float>::value || !(d2 >= s.t2_cut)) {
            T gx, gy;
            contact_force<T>(dx, dy, d2, dist_min, gx, gy);
            fx[a] = gx + fx[a]; fy[a] = gy + fy[a];
            fx[b] = -gx + fx[b]; fy[b] = -gy + fy[b];
          }
        }
      }
    }
#pragma unroll
    for (int i = 0; i < N; ++i) {
      if (!movable(i)) continue;
      integrate_agent<T>(px[i], py[i], vx[i], vy[i], fx[i], fy[i], max_speed);
    }
  }

  __device__ __forceinline__ static void goal_color(int g, T *c) {
    const T hi = SC == kReference ? (T)0.75 : (T)0.65, lo = SC == kReference ? (T)0.25 : (T)0.15;
    c[0] = g < 0 ? (T)0 : (g == 0 ? hi : lo);
    c[1] = g < 0 ? (T)0 : (g == 1 ? hi : lo);
    c[2] = g < 0 ? (T)0 : (g == 2 ? hi : lo);
  }

  // Observation of agent i -> row[0..D).  comm_other: message of the other agent (reference only).
  template <typename Row>
  __device__ __forceinline__ void obs_row(int i, Row row, const T *comm_other) const {
    if (SC == kSpread) {
      row[0] = vx[i]; row[1] = vy[i]; row[2] = px[i]; row[3] = py[i];
#pragma unroll
      for (int l = 0; l < L; ++l) {
        row[4 + 2 * l] = lx[l] - px[i];
        row[5 + 2 * l] = ly[l] - py[i];
      }
    } else {
      row[0] = vx[i]; row[1] = vy[i];
#pragma unroll
      for (int l = 0; l < L; ++l) {
        row[2 + 2 * l] = lx[l] - px[i];
        row[3 + 2 * l] = ly[l] - py[i];
      }
      T c[3];
      goal_color(goal[i], c);
      row[8] = c[0]; row[9] = c[1]; row[10] = c[2];
      if (SC == kReference) {
#pragma unroll
        for (int k = 0; k < 10; ++k) row[11 + k] = comm_other[k];
      }
    }
  }

  // Rewards (per agent, world.collaborative = False: experiments/scenarios.py:171) and the
  // integer channels of simple_spread's benchmark_data.
  __device__ __forceinline__ void reward(T *rew, int *coll, int &occupied, T &min_dists, const EnvState<T> &s) const {
    occupied = 0;
    min_dists = (T)0;
    if (SC == kSpread) {
      T base = (T)0;
#pragma unroll
      for (int l = 0; l < L; ++l) {
        // min_a sqrt(d2) == sqrt(min_a d2): sqrt is monotone and correctly rounded
        T m2 = (T)0;
#pragma unroll
        for (int a = 0; a < N; ++a) {
          const T dx = px[a] - lx[l], dy = py[a] - ly[l];
          const T d2 = sq2<T>(dx, dy);
          m2 = (a == 0) ? d2 : (d2 < m2 ? d2 : m2);
        }
        const T m = sqrt(m2);
        base -= m;
        min_dists += m;
        occupied += (m2 < s.t2_occ) ? 1 : 0;
      }
      bool hit[N][N];
#pragma unroll
      for (int a = 0; a < N; ++a) {
        {  // upstream also tests the agent against itself: dist 0 < dist_min, a constant -1 (NaN: no hit)
          const T zx = px[a] - px[a], zy = py[a] - py[a];
          hit[a][a] = sq2<T>(zx, zy) < s.t2_coll;
        }
#pragma unroll
        for (int b = a + 1; b < N; ++b) {
          const T dx = px[a] - px[b], dy = py[a] - py[b];
          const bool h = sq2<T>(dx, dy) < s.t2_coll;  // == sqrt(d2) < dist_min, exactly
          hit[a][b] = h; hit[b][a] = h;
        }
      }
#pragma unroll
      for (int i = 0; i < N; ++i) {
        T r = base;
        int c = 0;
#pragma unroll
        for (int a = 0; a < N; ++a)
          if (hit[a][i]) { r -= (T)1; ++c; }
        rew[i] = r;
        coll[i] = c;
      }
    } else if (SC == kReference) {
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const int g = goal[i];
        const T gx = g == 0 ? lx[0] : (g == 1 ? lx[1] : lx[2]);
        const T gy = g == 0 ? ly[0] : (g == 1 ? ly[1] : ly[2]);
        const T dx = px[1 - i] - gx, dy = py[1 - i] - gy;
        rew[i] = g < 0 ? (T)0 : -sq2<T>(dx, dy);
        coll[i] = 0;
      }
    } else {
      const int g = goal[0];
      const T gx = g == 0 ? lx[0] : (g == 1 ? lx[1] : lx[2]);
      const T gy = g == 0 ? ly[0] : (g == 1 ? ly[1] : ly[2]);
      const T dx = px[1] - gx, dy = py[1] - gy;
      rew[0] = rew[1] = -sq2<T>(dx, dy);
      coll[0] = coll[1] = 0;
    }
  }
};

}  // namespace mpe
