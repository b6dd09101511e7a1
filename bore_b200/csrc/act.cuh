// Element-wise layer activations (BORE_ACT_*) of every kernel that evaluates a net: forward, and the
// derivative wrt the pre-activation expressed through the layer OUTPUT h -- the only value the kernels
// keep, as TF's ReluGrad / EluGrad / SeluGrad / SigmoidGrad / TanhGrad kernels take it.  Only activations
// whose derivative is a function of h belong here (DESIGN.md, "Activations").
//
// The fp32 forms restate TensorFlow 2.5: selu and elu take expm1f where TF writes exp(a) - 1; softplus
// keeps softplus_op.h's thresholds; hard_sigmoid rounds the product and the sum separately, as the
// Keras backend's multiply and add ops do (no FMA contraction).
//
// Every kernel comes in two builds, selected at launch from the net's codes: EXT = false handles the five
// codes up to BORE_ACT_TANH with exactly the switch they always had, so that existing nets run the same
// instructions in the same registers; EXT = true adds the codes above it.
#pragma once
#include "common.cuh"

namespace {

constexpr float kSeluScale = 1.0507009873554805f;       // relu_op_functor.h Selu / SeluGrad
constexpr float kSeluScaleAlpha = 1.7580993408473768f;  // scale * alpha, as TF rounds it
constexpr float kSoftplusThreshold = -0x1.be2804p+3f;   // log(FLT_EPSILON) + 2 = -13.942385 (softplus_op.h)

__device__ __forceinline__ float act_fwd_ext(int a, float v) {
  switch (a) {
    case BORE_ACT_SELU: return v > 0.f ? kSeluScale * v : kSeluScaleAlpha * expm1f(v);
    case BORE_ACT_SOFTPLUS:
      return v > -kSoftplusThreshold ? v : (v < kSoftplusThreshold ? expf(v) : logf(expf(v) + 1.f));
    case BORE_ACT_SOFTSIGN: return v / (fabsf(v) + 1.f);
    case BORE_ACT_HARD_SIGMOID: return fminf(fmaxf(__fadd_rn(__fmul_rn(v, 0.2f), 0.5f), 0.f), 1.f);
    case BORE_ACT_EXPONENTIAL: return expf(v);
    default: return v;
  }
}
template <bool EXT>
__device__ __forceinline__ float act_fwd(int a, float v) {
  if (EXT && a > BORE_ACT_TANH) return act_fwd_ext(a, v);
  switch (a) {
    case BORE_ACT_RELU: return fmaxf(v, 0.f);
    case BORE_ACT_ELU: return v > 0.f ? v : expm1f(v);
    case BORE_ACT_SIGMOID: return 1.f / (1.f + expf(-v));
    case BORE_ACT_TANH: return tanhf(v);
    default: return v;
  }
}

// d act / d pre-activation from the output h.  softplus, softsign and hard_sigmoid differ from TF's
// features-based gradients by rounding (and hard_sigmoid at its two edges); DESIGN.md bounds how much.
__device__ __forceinline__ float act_bwd_ext(int a, float h) {
  switch (a) {
    case BORE_ACT_SELU: return h < 0.f ? h + kSeluScaleAlpha : kSeluScale;
    case BORE_ACT_SOFTPLUS: return -expm1f(-h);
    case BORE_ACT_SOFTSIGN: { const float t = 1.f - fabsf(h); return t * t; }
    case BORE_ACT_HARD_SIGMOID: return h > 0.f && h < 1.f ? 0.2f : 0.f;
    case BORE_ACT_EXPONENTIAL: return h;
    default: return 1.f;
  }
}
template <bool EXT>
__device__ __forceinline__ float act_bwd(int a, float h) {
  if (EXT && a > BORE_ACT_TANH) return act_bwd_ext(a, h);
  switch (a) {
    case BORE_ACT_RELU: return h > 0.f ? 1.f : 0.f;
    case BORE_ACT_ELU: return h > 0.f ? 1.f : h + 1.f;
    case BORE_ACT_SIGMOID: return h * (1.f - h);
    case BORE_ACT_TANH: return 1.f - h * h;
    default: return 1.f;
  }
}

// does a net need the EXT build of the kernels
inline bool acts_ext(const int *act, int n) {
  for (int l = 0; l < n; ++l)
    if (act[l] > BORE_ACT_TANH) return true;
  return false;
}

}  // namespace
