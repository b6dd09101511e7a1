// Device helpers shared by the training kernels (fit.cu: FP32 FFMA; fit_mma.cu: 3xTF32 tensor pipe).
#pragma once
#include "common.cuh"
#include "act.cuh"
#include "opt.cuh"

namespace {

__device__ __forceinline__ float stable_sigmoid(float u) {
  if (u >= 0.f) return 1.f / (1.f + expf(-u));
  const float e = expf(u);
  return e / (1.f + e);
}

__device__ __forceinline__ float block_sum(float v, float *red) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  float t = 0.f;
  const int nw = blockDim.x >> 5;
  for (int i = 0; i < nw; ++i) t += red[i];
  return t;
}

// e / n for 0 <= e < 2^20 through a precomputed reciprocal (inv = 1.f / n): exact, the offset .5
// keeps the product away from integer boundaries
__device__ __forceinline__ int fdiv(int e, float inv) { return __float2int_rz(((float)e + 0.5f) * inv); }

}  // namespace
