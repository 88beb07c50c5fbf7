// The LSTM cell's activations of the fp32 FFMA actor (actor_kernels.cu), shared with its backward
// (actor_grad_kernels.cu) so that the backward recomputes the forward's gates and relu masks bit for bit.
#pragma once

namespace mpe {

__device__ __forceinline__ float sigmoid_f(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }
__device__ __forceinline__ float tanh_f(float x) { return 1.0f - __fdividef(2.0f, 1.0f + __expf(2.0f * x)); }

}  // namespace mpe
