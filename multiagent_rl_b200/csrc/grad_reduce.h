// Weight gradients as sums over rows (grad_reduce.cu), shared by the critic's and the actor's backward: every weight
// gradient of both networks is sum_r A[r][m] B[r][k] over the (sample, agent) rows a backward kernel leaves in its
// workspace, plus the bias sum_r A[r][m].  Two launches, no floating-point atomics, every sum in an order fixed by
// the shapes alone:
//   1. k_grad_partial - CTA (tile, chunk) sums the rows of one chunk of a fixed chunking into its own slot of the
//      partial buffer;
//   2. k_grad_sum - the chunk partials added in chunk order into the caller's tensors.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace mpe {

// One sum over rows: out[m][k] = sum_r A[r][m] B[r][k] (k < kk), bias[m] = sum_r A[r][m], m < mm <= 64, kk <= 64.
struct GradTile {
  const float *a, *b;
  int64_t rows;
  int a_stride, b_stride, mm, kk;
  int out, ldo, bias;  // offsets into one chunk's partial vector; bias < 0: none
};
constexpr int kMaxTiles = 12;
struct GradTiles {
  GradTile t[kMaxTiles];
  int nchunk, nout;
};
// One caller tensor: n floats of the chunk-summed partial vector from offset src.
struct GradSeg {
  float *dst;
  int src, n;  // src < 0: zeros (a head with no upstream gradient)
};
constexpr int kMaxSegs = 16;  // the pointers of ActorGrads (CriticGrads has 10)
struct GradSegs {
  GradSeg s[kMaxSegs];
  int nseg, nchunk, nout;
};

// Chunks of the row range: at least kChunkRows rows each, at most kMaxChunks of them.
constexpr int kMaxChunks = 64, kChunkRows = 64;
inline int grad_chunks(int64_t rows) {
  const int n = (int)(rows < (int64_t)kMaxChunks * kChunkRows ? (rows + kChunkRows - 1) / kChunkRows : kMaxChunks);
  return n < 1 ? 1 : n;
}

// Launches both kernels on `st` for the first `ntiles` tiles of `tiles` into the non-empty `segs`; `partial` holds
// tiles.nchunk * tiles.nout floats.  `segs.nseg == 0` launches nothing.
cudaError_t launch_grad_reduce(GradTiles tiles, int ntiles, GradSegs segs, float *partial, cudaStream_t st);

}  // namespace mpe
