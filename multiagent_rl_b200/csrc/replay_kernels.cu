// Device-resident replay ring (SURVEY section 8f "next" row 1): rls/replay_buffer.py:9-91 (ReplayBuffer.add /
// make_index / sample_index / _encode_sample) and the transition tuple built at experiments/run.py:46,52
// (obs_n, action_n_env, rew_shared = sum(rew_n), new_obs_n, float(done)), for B env instances at a time.
// A transition is one contiguous record of the ring (replay_launch.h); add is a streaming copy into consecutive
// records, sample a gather of whole records.
#include "replay_launch.h"

#include "common.cuh"
#include "launch.h"

namespace mpe {

// add: ring slots (head + b) % capacity are contiguous apart from one wrap, so the host splits the batch at the wrap and
// a segment fills CONSECUTIVE records.  A block assembles `rpb` records in shared memory (256 / rpb threads per row:
// coalesced reads of the caller's obs / obs_next rows, the action bytes, the shared reward) and writes them out as one
// contiguous, 16 B-vectorised span - writing the record fields straight from the source layout (8 B stores into
// alternating 120 B halves of 256 B records) reached 0.54 of HBM, separate arrays 0.95 for the add but 0.47 for sample.
template <int V>  // floats per vector of the observation copies: 2 (R even, 8 B aligned sources) or 1
__global__ void __launch_bounds__(256) k_replay_add(ReplayDev r, int64_t slot0, int64_t rows, int rpb, const float *__restrict__ obs,
                                                    const int32_t *__restrict__ act_u, const int32_t *__restrict__ act_c,
                                                    const float *__restrict__ rew, const float *__restrict__ obs_next,
                                                    const float *__restrict__ done) {
  extern __shared__ __align__(16) unsigned char tile[];
  const int R = r.N * r.D, RV = R / V, rec = (int)r.rec_bytes;
  const int dj = 256 / RV, dc = 256 - dj * RV;  // (row, column) of a flat vector index advance by this per 256 threads
  for (int64_t b0 = (int64_t)blockIdx.x * rpb; b0 < rows; b0 += (int64_t)gridDim.x * rpb) {
    const int nrows = (int)((rows - b0) < rpb ? (rows - b0) : rpb);
    // phase 1: the block's rows of obs / obs_next are one contiguous span each: flat, coalesced reads; the shared-memory
    // address of an element follows from its (row, column), advanced incrementally
    {
      int row = threadIdx.x / RV, c = threadIdx.x - row * RV;
      const float *so = obs + b0 * R, *sn = obs_next + b0 * R;
      for (int e = threadIdx.x; e < nrows * RV; e += 256, row += dj, c += dc) {
        if (c >= RV) { c -= RV; ++row; }
        unsigned char *rp = tile + row * rec;
        if (V == 2) {
          reinterpret_cast<float2 *>(rp)[c] = reinterpret_cast<const float2 *>(so)[e];
          reinterpret_cast<float2 *>(rp + r.off_next())[c] = reinterpret_cast<const float2 *>(sn)[e];
        } else {
          reinterpret_cast<float *>(rp)[c] = so[e];
          reinterpret_cast<float *>(rp + r.off_next())[c] = sn[e];
        }
      }
    }
    for (int e = threadIdx.x; e < nrows * r.N; e += 256) {
      const int row = e / r.N, n = e - row * r.N;
      tile[row * rec + r.off_au() + n] = (unsigned char)(int8_t)act_u[b0 * r.N + e];
      tile[row * rec + r.off_ac() + n] = act_c != nullptr ? (unsigned char)(int8_t)act_c[b0 * r.N + e] : (unsigned char)0;
    }
    for (int row = threadIdx.x; row < nrows; row += 256) {
      float s = 0.0f;  // rew_shared = np.sum(rew_n) (experiments/run.py:46), agent order
      for (int n = 0; n < r.N; ++n) s += rew[(b0 + row) * r.N + n];
      *reinterpret_cast<float *>(tile + row * rec + r.off_rew()) = s;
      *reinterpret_cast<float *>(tile + row * rec + r.off_done()) = done != nullptr ? done[b0 + row] : 0.0f;
    }
    __syncthreads();
    // phase 2: nrows consecutive records = one contiguous span of the ring, 16 B per lane
    uint4 *dst = reinterpret_cast<uint4 *>(r.ring + (slot0 + b0) * r.rec_bytes);
    const uint4 *src = reinterpret_cast<const uint4 *>(tile);
    for (int v = threadIdx.x; v < nrows * (rec / 16); v += 256) dst[v] = src[v];
    __syncthreads();
  }
}

// add for T steps of a rollout at once: k_replay_add's record assembly on a (block, step) grid.  Step t's obs_t is
// obs0 for t = 0 and obs_next[t - 1] after that (within one episode the observation an actor acts on is the one the
// previous step returned); transition `first + t * B + b` of the call lands in ring slot (head + that) % capacity.
// Transitions before `keep_from` would be overwritten by a later transition of the same call: they are skipped, so
// that no two blocks of one launch write the same slot.  A block's records are one ring span apart from one wrap.
template <int V>
__global__ void __launch_bounds__(256) k_replay_add_steps(ReplayDev r, int64_t head, int64_t B, int T, int64_t first,
                                                          int64_t keep_from, int rpb, const float *__restrict__ obs0,
                                                          const float *__restrict__ obs_next, const int32_t *__restrict__ act_u,
                                                          const int32_t *__restrict__ act_c, const float *__restrict__ rew) {
  extern __shared__ __align__(16) unsigned char tile[];
  const int R = r.N * r.D, RV = R / V, rec = (int)r.rec_bytes, VPR = rec / 16;
  const int dj = 256 / RV, dc = 256 - dj * RV;
  for (int t = blockIdx.y; t < T; t += gridDim.y) {
    const float *so_t = t == 0 ? obs0 : obs_next + (int64_t)(t - 1) * B * R, *sn_t = obs_next + (int64_t)t * B * R;
    const int64_t g_t = first + (int64_t)t * B;  // call-wide index of env 0's transition of step t
    for (int64_t bb = (int64_t)blockIdx.x * rpb; bb < B; bb += (int64_t)gridDim.x * rpb) {
      const int64_t skip = keep_from - (g_t + bb), end = (B - bb) < rpb ? (B - bb) : rpb;
      if (skip >= end) continue;  // uniform per block
      const int64_t b0 = skip > 0 ? bb + skip : bb;
      const int nrows = (int)(bb + end - b0);
      {
        int row = threadIdx.x / RV, c = threadIdx.x - row * RV;
        const float *so = so_t + b0 * R, *sn = sn_t + b0 * R;
        for (int e = threadIdx.x; e < nrows * RV; e += 256, row += dj, c += dc) {
          if (c >= RV) { c -= RV; ++row; }
          unsigned char *rp = tile + row * rec;
          if (V == 2) {
            reinterpret_cast<float2 *>(rp)[c] = reinterpret_cast<const float2 *>(so)[e];
            reinterpret_cast<float2 *>(rp + r.off_next())[c] = reinterpret_cast<const float2 *>(sn)[e];
          } else {
            reinterpret_cast<float *>(rp)[c] = so[e];
            reinterpret_cast<float *>(rp + r.off_next())[c] = sn[e];
          }
        }
      }
      const int64_t a0 = (int64_t)t * B * r.N + b0 * r.N;
      for (int e = threadIdx.x; e < nrows * r.N; e += 256) {
        const int row = e / r.N, n = e - row * r.N;
        tile[row * rec + r.off_au() + n] = (unsigned char)(int8_t)act_u[a0 + e];
        tile[row * rec + r.off_ac() + n] = act_c != nullptr ? (unsigned char)(int8_t)act_c[a0 + e] : (unsigned char)0;
      }
      for (int row = threadIdx.x; row < nrows; row += 256) {
        float s = 0.0f;  // rew_shared = np.sum(rew_n) (experiments/run.py:46), agent order
        for (int n = 0; n < r.N; ++n) s += rew[a0 + (int64_t)row * r.N + n];
        *reinterpret_cast<float *>(tile + row * rec + r.off_rew()) = s;
        *reinterpret_cast<float *>(tile + row * rec + r.off_done()) = 0.0f;
      }
      __syncthreads();
      // the first n1 records end at the ring's last slot, the rest continue at slot 0
      const int64_t s0 = (head + g_t + b0) % r.capacity;
      const int n1v = (int)((r.capacity - s0) < nrows ? (r.capacity - s0) : nrows) * VPR;
      uint4 *dst0 = reinterpret_cast<uint4 *>(r.ring + s0 * r.rec_bytes), *dst1 = reinterpret_cast<uint4 *>(r.ring);
      const uint4 *src = reinterpret_cast<const uint4 *>(tile);
      for (int v = threadIdx.x; v < nrows * VPR; v += 256) {
        if (v < n1v) dst0[v] = src[v]; else dst1[v - n1v] = src[v];
      }
      __syncthreads();
    }
  }
}

// uniform indices with replacement: random.randint(0, len - 1) per sample (rls/replay_buffer.py:51-52)
__global__ void __launch_bounds__(256) k_replay_make_index(int64_t size, int64_t batch, uint64_t seed, uint64_t counter,
                                                           int64_t *__restrict__ idx) {
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < batch; j += (int64_t)gridDim.x * blockDim.x) {
    const uint4 rr = philox_raw(seed, (uint64_t)j, (uint32_t)counter, kDomainReplay,
                                (uint32_t)(counter >> 32) & 0xFFFFu);
    idx[j] = (int64_t)__umul64hi(((uint64_t)rr.x << 32) | rr.y, (uint64_t)size);
  }
}

// gather `batch` transitions by index, element-parallel over the flattened [batch][R] output (8 B vectors when R is
// even): every lane moves data although one transition is only R * 4 = 120 B (simple_spread N = 3), and a warp's stores
// are one aligned 256 B span.  (Measured and not kept: 16 lanes per row with shift / mask indexing instead of the two
// divisions per element - 0.37 of HBM, with 4 rows in flight per lane group 0.30, against 0.47 for this form.)
template <int V>
__global__ void __launch_bounds__(256) k_replay_gather(ReplayDev r, int64_t size, int64_t batch, const int64_t *__restrict__ idx,
                                                       float *__restrict__ obs, float *__restrict__ act_onehot,
                                                       float *__restrict__ rew, float *__restrict__ obs_next,
                                                       float *__restrict__ done) {
  const int R = r.N * r.D, RV = R / V, A = r.A0 + r.A1;
  const int64_t total = batch * RV;
  // (row, column) of flat element i advance incrementally with the grid stride: two divisions per THREAD, none per element
  const int64_t stride = (int64_t)gridDim.x * blockDim.x, i0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t dj = stride / RV;
  const int dc = (int)(stride - dj * RV);
  int64_t j = i0 / RV;
  int c = (int)(i0 - j * RV);
  for (int64_t i = i0; i < total; i += stride, j += dj, c += dc) {
    if (c >= RV) { c -= RV; ++j; }
    // list indexing of ReplayBuffer._storage[i] (rls/replay_buffer.py:42): negative indices count from the end;
    // anything still outside [0, size) is clamped so that a stale index can never read outside the ring
    int64_t slot = idx[j];
    if (slot < 0) slot += size;
    slot = slot < 0 ? 0 : (slot >= size ? size - 1 : slot);
    const unsigned char *rec = r.ring + slot * r.rec_bytes;  // the whole transition: one contiguous record
    if (V == 2) {
      if (obs != nullptr) reinterpret_cast<float2 *>(obs + j * R)[c] = reinterpret_cast<const float2 *>(rec)[c];
      if (obs_next != nullptr)
        reinterpret_cast<float2 *>(obs_next + j * R)[c] = reinterpret_cast<const float2 *>(rec + r.off_next())[c];
    } else {
      if (obs != nullptr) obs[j * R + c] = reinterpret_cast<const float *>(rec)[c];
      if (obs_next != nullptr) obs_next[j * R + c] = reinterpret_cast<const float *>(rec + r.off_next())[c];
    }
    if (act_onehot != nullptr)
      for (int e = c; e < r.N * A; e += RV) {
        const int n = e / A, a = e - n * A;
        const int u = reinterpret_cast<const int8_t *>(rec + r.off_au())[n], cc = reinterpret_cast<const int8_t *>(rec + r.off_ac())[n];
        act_onehot[j * r.N * A + e] = (a < r.A0 ? a == u : a - r.A0 == cc) ? 1.0f : 0.0f;
      }
    if (c == 0) {
      if (rew != nullptr) rew[j] = *reinterpret_cast<const float *>(rec + r.off_rew());
      if (done != nullptr) done[j] = *reinterpret_cast<const float *>(rec + r.off_done());
    }
  }
}

// gather through shared memory (the mirror image of k_replay_add): a block pulls `rpb` sampled records into a tile with
// 16 B loads (16 lanes = one 256 B record = one DRAM burst), then writes every output array as a contiguous, coalesced
// span - consecutive sampled transitions are adjacent rows of obs / obs_next / act_onehot / rew / done.
template <int V>
__global__ void __launch_bounds__(256) k_replay_gather_tile(ReplayDev r, int64_t size, int64_t batch, int rpb,
                                                            const int64_t *__restrict__ idx, float *__restrict__ obs,
                                                            float *__restrict__ act_onehot, float *__restrict__ rew,
                                                            float *__restrict__ obs_next, float *__restrict__ done) {
  extern __shared__ __align__(16) unsigned char tile[];
  const int R = r.N * r.D, RV = R / V, rec = (int)r.rec_bytes, VPR = rec / 16, A = r.A0 + r.A1, NA = r.N * A;
  const int dj1 = 256 / VPR, dc1 = 256 - dj1 * VPR, dj2 = 256 / RV, dc2 = 256 - dj2 * RV;
  for (int64_t j0 = (int64_t)blockIdx.x * rpb; j0 < batch; j0 += (int64_t)gridDim.x * rpb) {
    const int nrows = (int)((batch - j0) < rpb ? (batch - j0) : rpb);
    {  // phase 1: whole records, 16 B per lane
      int row = threadIdx.x / VPR, k = threadIdx.x - row * VPR;
      for (int v = threadIdx.x; v < nrows * VPR; v += 256, row += dj1, k += dc1) {
        if (k >= VPR) { k -= VPR; ++row; }
        // list indexing of ReplayBuffer._storage[i] (rls/replay_buffer.py:42): negative indices count from the end;
        // anything still outside [0, size) is clamped so that a stale index can never read outside the ring
        int64_t slot = idx[j0 + row];
        if (slot < 0) slot += size;
        slot = slot < 0 ? 0 : (slot >= size ? size - 1 : slot);
        reinterpret_cast<uint4 *>(tile + row * rec)[k] = reinterpret_cast<const uint4 *>(r.ring + slot * r.rec_bytes)[k];
      }
    }
    __syncthreads();
    {  // phase 2: contiguous output spans
      int row = threadIdx.x / RV, c = threadIdx.x - row * RV;
      for (int e = threadIdx.x; e < nrows * RV; e += 256, row += dj2, c += dc2) {
        if (c >= RV) { c -= RV; ++row; }
        const unsigned char *rp = tile + row * rec;
        if (V == 2) {
          if (obs != nullptr) reinterpret_cast<float2 *>(obs + j0 * R)[e] = reinterpret_cast<const float2 *>(rp)[c];
          if (obs_next != nullptr) reinterpret_cast<float2 *>(obs_next + j0 * R)[e] = reinterpret_cast<const float2 *>(rp + r.off_next())[c];
        } else {
          if (obs != nullptr) obs[j0 * R + e] = reinterpret_cast<const float *>(rp)[c];
          if (obs_next != nullptr) obs_next[j0 * R + e] = reinterpret_cast<const float *>(rp + r.off_next())[c];
        }
      }
      if (act_onehot != nullptr)
        for (int e = threadIdx.x; e < nrows * NA; e += 256) {
          const int rw = e / NA, x = e - rw * NA, n = x / A, a = x - n * A;
          const unsigned char *rp = tile + rw * rec;
          const int u = reinterpret_cast<const int8_t *>(rp + r.off_au())[n], cc = reinterpret_cast<const int8_t *>(rp + r.off_ac())[n];
          act_onehot[j0 * NA + e] = (a < r.A0 ? a == u : a - r.A0 == cc) ? 1.0f : 0.0f;
        }
      for (int rw = threadIdx.x; rw < nrows; rw += 256) {
        if (rew != nullptr) rew[j0 + rw] = *reinterpret_cast<const float *>(tile + rw * rec + r.off_rew());
        if (done != nullptr) done[j0 + rw] = *reinterpret_cast<const float *>(tile + rw * rec + r.off_done());
      }
    }
    __syncthreads();
  }
}

static unsigned grid_for(int64_t total) {
  const int64_t blocks = (total + 255) / 256, cap = (int64_t)sm_count(current_device()) * 32;
  return (unsigned)(blocks < cap ? (blocks > 0 ? blocks : 1) : cap);
}

cudaError_t launch_replay_add(const ReplayDev &r, int64_t head, int64_t B, const float *obs, const int32_t *act_u,
                              const int32_t *act_c, const float *rew, const float *obs_next, const float *done,
                              cudaStream_t st) {
  if (B <= 0) return cudaSuccess;
  const int64_t R = (int64_t)r.N * r.D;
  int rpb = 128;  // records per block (32 KB of shared memory at 256 B per record)
  while (rpb > 1 && (int64_t)rpb * r.rec_bytes > 32 * 1024) rpb >>= 1;
  if (r.rec_bytes > kReplayMaxRecordBytes) return cudaErrorInvalidValue;
  const int64_t cap = (int64_t)sm_count(current_device()) * 16;
  int64_t row0 = 0;
  while (row0 < B) {  // at most capacity rows per segment; a batch larger than the ring wraps more than once
    const int64_t slot0 = (head + row0) % r.capacity;
    const int64_t rows = (B - row0) < (r.capacity - slot0) ? (B - row0) : (r.capacity - slot0);
    const int64_t blocks = (rows + rpb - 1) / rpb;
    const unsigned grid = (unsigned)(blocks < cap ? blocks : cap);
    const size_t sm = (size_t)rpb * r.rec_bytes;
    const uintptr_t al = reinterpret_cast<uintptr_t>(obs + row0 * R) | reinterpret_cast<uintptr_t>(obs_next + row0 * R);
    if (R % 2 == 0 && (al & 7) == 0)
      k_replay_add<2><<<grid, 256, sm, st>>>(r, slot0, rows, rpb, obs + row0 * R, act_u + row0 * r.N,
                                             act_c != nullptr ? act_c + row0 * r.N : nullptr, rew + row0 * r.N,
                                             obs_next + row0 * R, done != nullptr ? done + row0 : nullptr);
    else
      k_replay_add<1><<<grid, 256, sm, st>>>(r, slot0, rows, rpb, obs + row0 * R, act_u + row0 * r.N,
                                             act_c != nullptr ? act_c + row0 * r.N : nullptr, rew + row0 * r.N,
                                             obs_next + row0 * R, done != nullptr ? done + row0 : nullptr);
    row0 += rows;
  }
  return cudaGetLastError();
}

cudaError_t launch_replay_add_steps(const ReplayDev &r, int64_t head, int64_t B, int32_t T, int64_t first,
                                    int64_t keep_from, const float *obs0, const float *obs_next, const int32_t *act_u,
                                    const int32_t *act_c, const float *rew, cudaStream_t st) {
  if (B <= 0 || T <= 0) return cudaSuccess;
  if (r.rec_bytes > kReplayMaxRecordBytes) return cudaErrorInvalidValue;
  int rpb = 128;  // records per block, as launch_replay_add
  while (rpb > 1 && (int64_t)rpb * r.rec_bytes > 32 * 1024) rpb >>= 1;
  const int64_t blocks = (B + rpb - 1) / rpb, cap = (int64_t)sm_count(current_device()) * 16;
  const dim3 grid((unsigned)(blocks < cap ? blocks : cap), (unsigned)(T < 65535 ? T : 65535));
  const size_t sm = (size_t)rpb * r.rec_bytes;
  const bool v2 = (int64_t)r.N * r.D % 2 == 0 &&
                  ((reinterpret_cast<uintptr_t>(obs0) | reinterpret_cast<uintptr_t>(obs_next)) & 7) == 0;
  if (v2)
    k_replay_add_steps<2><<<grid, 256, sm, st>>>(r, head, B, T, first, keep_from, rpb, obs0, obs_next, act_u, act_c, rew);
  else
    k_replay_add_steps<1><<<grid, 256, sm, st>>>(r, head, B, T, first, keep_from, rpb, obs0, obs_next, act_u, act_c, rew);
  return cudaGetLastError();
}

cudaError_t launch_replay_make_index(int64_t size, int64_t batch, uint64_t seed, uint64_t counter, int64_t *idx,
                                     cudaStream_t st) {
  if (batch <= 0) return cudaSuccess;
  k_replay_make_index<<<grid_for(batch), 256, 0, st>>>(size, batch, seed, counter, idx);
  return cudaGetLastError();
}

cudaError_t launch_replay_gather(const ReplayDev &r, int64_t size, int64_t batch, const int64_t *idx, float *obs, float *act_onehot,
                                 float *rew, float *obs_next, float *done, cudaStream_t st) {
  if (batch <= 0) return cudaSuccess;
  const int R = r.N * r.D;
  const bool v2 = (R % 2 == 0) && ((reinterpret_cast<uintptr_t>(obs) | reinterpret_cast<uintptr_t>(obs_next)) & 7) == 0;
  int rpb = 64;  // records per block (16 KB of shared memory at 256 B per record; measured 128: 0.67, 64: 0.75, 32: 0.64 of HBM)
  while (rpb > 1 && (int64_t)rpb * r.rec_bytes > 16 * 1024) rpb >>= 1;
  if (r.rec_bytes <= 16 * 1024) {
    const int64_t blocks = (batch + rpb - 1) / rpb, cap = (int64_t)sm_count(current_device()) * 16;
    const unsigned grid = (unsigned)(blocks < cap ? blocks : cap);
    const size_t sm = (size_t)rpb * r.rec_bytes;
    if (v2)
      k_replay_gather_tile<2><<<grid, 256, sm, st>>>(r, size, batch, rpb, idx, obs, act_onehot, rew, obs_next, done);
    else
      k_replay_gather_tile<1><<<grid, 256, sm, st>>>(r, size, batch, rpb, idx, obs, act_onehot, rew, obs_next, done);
    return cudaGetLastError();
  }
  if (v2)  // records too large for a tile: element-parallel gather straight from the ring
    k_replay_gather<2><<<grid_for(batch * (R / 2)), 256, 0, st>>>(r, size, batch, idx, obs, act_onehot, rew, obs_next, done);
  else
    k_replay_gather<1><<<grid_for(batch * R), 256, 0, st>>>(r, size, batch, idx, obs, act_onehot, rew, obs_next, done);
  return cudaGetLastError();
}

}  // namespace mpe
