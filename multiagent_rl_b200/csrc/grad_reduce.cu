// Row-sum reductions of the backward kernels (grad_reduce.h): critic_grad_kernels.cu and actor_grad_kernels.cu.
#include "grad_reduce.h"

namespace mpe {

// CTA (tile, chunk): 256 threads, thread (ty, tx) owns out[ty + 16 i][tx + 16 j]; rows are staged 32 at a time
__global__ void __launch_bounds__(256) k_grad_partial(GradTiles p, float *__restrict__ partial) {
  __shared__ float As[32][64], Bs[32][64];
  const GradTile &T = p.t[blockIdx.x];
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  const int64_t cs = (T.rows + p.nchunk - 1) / p.nchunk, r0 = (int64_t)blockIdx.y * cs;
  const int64_t r1 = r0 + cs < T.rows ? r0 + cs : T.rows;
  float acc[4][4] = {}, bacc = 0.0f;
  for (int64_t rb = r0; rb < r1; rb += 32) {
    __syncthreads();
    for (int i = tid; i < 32 * 64; i += 256) {
      const int rr = i >> 6, cc = i & 63;
      const int64_t row = rb + rr;
      As[rr][cc] = row < r1 && cc < T.mm ? T.a[row * T.a_stride + cc] : 0.0f;
      Bs[rr][cc] = row < r1 && cc < T.kk ? T.b[row * T.b_stride + cc] : 0.0f;
    }
    __syncthreads();
    const int nr = r1 - rb < 32 ? (int)(r1 - rb) : 32;
    for (int rr = 0; rr < nr; ++rr) {
      float av[4], bv[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { av[i] = As[rr][ty + 16 * i]; bv[i] = Bs[rr][tx + 16 * i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
      if (tid < 64) bacc += As[rr][tid];
    }
  }
  float *P = partial + (int64_t)blockIdx.y * p.nout;
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int m = ty + 16 * i, k = tx + 16 * j;
      if (m < T.mm && k < T.kk) P[T.out + m * T.ldo + k] = acc[i][j];
    }
  if (T.bias >= 0 && tid < T.mm) P[T.bias + tid] = bacc;
}

__global__ void __launch_bounds__(256) k_grad_sum(GradSegs p, const float *__restrict__ partial) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  for (int g = 0; g < p.nseg; ++g) {
    if (i < p.s[g].n) {
      float v = 0.0f;
      if (p.s[g].src >= 0)
        for (int c = 0; c < p.nchunk; ++c) v += partial[(int64_t)c * p.nout + p.s[g].src + i];
      p.s[g].dst[i] = v;
      return;
    }
    i -= p.s[g].n;
  }
}

cudaError_t launch_grad_reduce(GradTiles tiles, int ntiles, GradSegs segs, float *partial, cudaStream_t st) {
  if (segs.nseg == 0) return cudaSuccess;
  k_grad_partial<<<dim3(ntiles, tiles.nchunk), 256, 0, st>>>(tiles, partial);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  segs.nchunk = tiles.nchunk;
  segs.nout = tiles.nout;
  int total = 0;
  for (int i = 0; i < segs.nseg; ++i) total += segs.s[i].n;
  k_grad_sum<<<(total + 255) / 256, 256, 0, st>>>(segs, partial);
  return cudaGetLastError();
}

}  // namespace mpe
