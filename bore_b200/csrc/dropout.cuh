// Keras Dropout between Dense layers (DESIGN.md, "Dropout"): the descriptor of a handle, the mask and the rule
// of TF 2.5's nn_ops.dropout_v2 with a number rate.  The only place that knows the mask layout.
//
// Mask: Philox4x32-10 (Random123).  Hidden layer l, unit j, sample position i of the minibatch, model m, step t
// (the model's Keras `iterations` before this step's increment):
//   counter = (t mod 2^32, t div 2^32, i, 65536 l + j div 4), key = (seed_l, m), w = output word j mod 4,
//   keep  <=>  (w >> 8) 2^-24 >= rate_l
// so one Philox call gives the keep bits of four consecutive units of one sample.
// Rule: forward  h~ = fl32(h scale) keep;  reverse  dL/dh = fl32(dL/dh~ keep) scale, times act'(h).
#pragma once
#include "common.cuh"
#include "act.cuh"

// The dropout of a fit launch, passed by value to the fit kernels (FitJob::drop, from the handle's
// bore_mlp_set_dropout).  All zeros: no dropout.
struct Dropout {
  float rate[BORE_MAX_LAYERS];   // hidden layer l (the output of Dense l): 0 = none
  float scale[BORE_MAX_LAYERS];  // fp32(1 / (1 - rate)), computed in double on the host: the kernels never divide
  uint32_t seed[BORE_MAX_LAYERS];
  int any;                       // some rate is > 0
};

namespace {

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r > 0) { k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
  }
  return c;
}

__device__ __forceinline__ uint32_t drop_bit(uint32_t w, float rate) {
  return __uint2float_rz(w >> 8) * 5.9604644775390625e-8f >= rate ? 1u : 0u;  // (exact: 24 bits times 2^-24)
}

// keep bits of units 4q .. 4q + 3 of sample i in hidden layer l (bit u: unit 4q + u)
__device__ __forceinline__ uint32_t drop_keep4(const Dropout &dp, int l, long long t, int i, int q, int m) {
  const uint4 w = philox4x32_10(make_uint4((uint32_t)t, (uint32_t)((unsigned long long)t >> 32), (uint32_t)i,
                                           (uint32_t)(65536 * l + q)),
                                dp.seed[l], (uint32_t)m);
  const float r = dp.rate[l];
  return drop_bit(w.x, r) | drop_bit(w.y, r) << 1 | drop_bit(w.z, r) << 2 | drop_bit(w.w, r) << 3;
}

// keep of unit j of sample i in hidden layer l
__device__ __forceinline__ bool drop_keep(const Dropout &dp, int l, long long t, int i, int j, int m) {
  return (drop_keep4(dp, l, t, i, j >> 2, m) >> (j & 3)) & 1u;
}

// forward: h~ = fl32(h scale) keep
__device__ __forceinline__ float drop_fwd(float h, bool keep, float scale) {
  return __fmul_rn(__fmul_rn(h, scale), keep ? 1.f : 0.f);
}

// act'(h) of a kept unit from h~ = fl32(h scale), the value the kernels keep in place of h.  Rounding is monotone and
// scale > 1, so h < 1 gives h~ < scale, h = 1 gives h~ = scale and h > 1 gives h~ > scale (the same at -1), and the
// sign of h is the sign of h~.  So every threshold of act' is tested exactly: hard_sigmoid's 0 < h < 1 as
// 0 < h~ < scale, relu / elu / selu on the sign, and the saturated h = +-1 of sigmoid, tanh and softsign is restored
// exactly.  Elsewhere h is fl32(h~ fp32(1 - rate)), within a few ulp of h: the smooth act' moves by as much.
template <bool EXT>
__device__ __forceinline__ float drop_act_bwd(int act, float hd, float scale, float rate) {
  if (EXT && act == BORE_ACT_HARD_SIGMOID) return hd > 0.f && hd < scale ? 0.2f : 0.f;
  return act_bwd<EXT>(act, fabsf(hd) == scale ? copysignf(1.f, hd) : __fmul_rn(hd, 1.f - rate));
}

// reverse: dL/du = fl32(fl32(g keep) scale) act'(h) with g = dL/dh~
template <bool EXT>
__device__ __forceinline__ float drop_bwd(int act, float g, float hd, bool keep, float scale, float rate) {
  return __fmul_rn(__fmul_rn(g, keep ? 1.f : 0.f), scale) * drop_act_bwd<EXT>(act, hd, scale, rate);
}

// the same for unit j of the four samples i0 .. i0 + 3 (the float4 epilogues of the FFMA kernels)
__device__ __forceinline__ float4 drop_fwd_unit4(const Dropout &dp, int l, long long t, int i0, int j, int m, float4 h) {
  const float s = dp.scale[l];
  return make_float4(drop_fwd(h.x, drop_keep(dp, l, t, i0, j, m), s), drop_fwd(h.y, drop_keep(dp, l, t, i0 + 1, j, m), s),
                     drop_fwd(h.z, drop_keep(dp, l, t, i0 + 2, j, m), s), drop_fwd(h.w, drop_keep(dp, l, t, i0 + 3, j, m), s));
}
template <bool EXT>
__device__ __forceinline__ float4 drop_bwd_unit4(const Dropout &dp, int l, long long t, int i0, int j, int m, int act,
                                                 float4 g, float4 hd) {
  const float s = dp.scale[l], r = dp.rate[l];
  return make_float4(drop_bwd<EXT>(act, g.x, hd.x, drop_keep(dp, l, t, i0, j, m), s, r),
                     drop_bwd<EXT>(act, g.y, hd.y, drop_keep(dp, l, t, i0 + 1, j, m), s, r),
                     drop_bwd<EXT>(act, g.z, hd.z, drop_keep(dp, l, t, i0 + 2, j, m), s, r),
                     drop_bwd<EXT>(act, g.w, hd.w, drop_keep(dp, l, t, i0 + 3, j, m), s, r));
}

}  // namespace
