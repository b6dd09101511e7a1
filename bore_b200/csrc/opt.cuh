// Keras optimizers (BORE_OPT_*) of every training kernel: the per-step scalars and the update of one
// parameter on the two fp32 slots every kernel keeps per parameter (adam_m / adam_v of the handles).
//
// Slots per kind (DESIGN.md, "Optimizers"):
//   Adam      m / v                     Adamax    m / v (v = the exponentially weighted infinity norm)
//   RMSprop   rms / mom (momentum > 0) or mg (centered), unused otherwise
//   Adagrad   accumulator / unused      Adadelta  accum_grad / accum_var
//   Nadam     m / v, and one fp32 scalar per model, the momentum cache (OptRun::cache)
// Padding parameters of the kernels have a zero gradient and zero slots: every rule leaves them exactly zero
// as long as eps > 0, which bore_*_set_optimizer_kind demands of every kind but Adam.
//
// Every fit kernel comes in two builds, selected at launch from the kind: OPT = false is Adam only, with the
// arithmetic and the instructions it always had; OPT = true adds the other kinds.
#pragma once
#include "common.cuh"

namespace {

// Nadam's momentum schedule: mu_t = beta_1 (1 - 0.5 * 0.96^(0.004 t))  (keras/optimizer_v2/nadam.py)
constexpr double kNadamDecayBase = 0.96, kNadamCacheDecay = 0.004;

// scalars of one step, the same for every parameter of a model
struct OptStep {
  float om1, om2;  // 1 - beta_1 (or 1 - rho), 1 - beta_2
  float alpha;     // Adam: lr sqrt(1 - beta_2^t) / (1 - beta_1^t); Adamax: lr / (1 - beta_1^t); else lr
  float cg, cm;    // Nadam: (1 - mu_t) / (1 - cache_t), mu_{t+1} / (1 - cache_t mu_{t+1})
  float vd;        // Nadam: 1 / (1 - beta_2^t)
};

// The optimizer state of one model inside a fit kernel: Keras `iterations`, beta^t as fp64 running products
// (one multiplication per step instead of two pow calls) and Nadam's momentum cache.
template <bool OPT>
struct OptRun {
  long long t;
  double p1, p2;  // beta_1^t (Nadam: 0.96^(0.004 t)), beta_2^t
  double f1;      // the factor of p1 (OPT only)
  float cache;    // Nadam's momentum cache (OPT only)

  __device__ __forceinline__ OptRun(const OptHyper &h, long long t0, const float *cache_dev) : t(t0) {
    f1 = OPT && h.kind == BORE_OPT_NADAM ? pow(kNadamDecayBase, kNadamCacheDecay) : (double)h.b1;
    p1 = pow(OPT ? f1 : (double)h.b1, (double)t0);
    p2 = pow((double)h.b2, (double)t0);
    cache = OPT ? *cache_dev : 1.f;
  }

  // the scalars that stay the same for every step (fit_mma.cu keeps them out of its loop)
  __device__ __forceinline__ static OptStep consts(const OptHyper &h) {
    OptStep s;
    s.om1 = 1.f - h.b1;
    s.om2 = 1.f - h.b2;
    s.alpha = s.cg = s.cm = s.vd = 0.f;
    return s;
  }

  // advance to the next step (Keras: t starts at 1): the scalars of s that depend on it
  __device__ __forceinline__ void advance(const OptHyper &h, OptStep &s) {
    t += 1;
    if (!OPT) {
      p1 *= (double)h.b1;
      p2 *= (double)h.b2;
      const float b1p = (float)p1, b2p = (float)p2;
      s.alpha = h.lr * sqrtf(1.f - b2p) / (1.f - b1p);
      return;
    }
    p1 *= f1;
    p2 *= (double)h.b2;
    switch (h.kind) {
      case BORE_OPT_ADAM: s.alpha = h.lr * sqrtf(1.f - (float)p2) / (1.f - (float)p1); break;
      case BORE_OPT_ADAMAX: s.alpha = h.lr / (1.f - (float)p1); break;
      case BORE_OPT_NADAM: {
        const float mu = h.b1 * (1.f - 0.5f * (float)p1), mu_next = h.b1 * (1.f - 0.5f * (float)(p1 * f1));
        cache *= mu;  // fp32, as Keras keeps its m_cache variable
        s.alpha = h.lr;
        s.cg = (1.f - mu) / (1.f - cache);
        s.cm = mu_next / (1.f - cache * mu_next);
        s.vd = 1.f / (1.f - (float)p2);
        break;
      }
      default: s.alpha = h.lr; break;
    }
  }

  // advance to the next step and give all its scalars
  __device__ __forceinline__ OptStep step(const OptHyper &h) {
    OptStep s = consts(h);
    advance(h, s);
    return s;
  }

  // written back by one thread at the end of the kernel
  __device__ __forceinline__ void store(long long *t_dev, float *cache_dev) const {
    *t_dev = t;
    if (OPT) *cache_dev = cache;
  }
};

__device__ __forceinline__ float sqrt_approx(float v) {
  float r;
  asm("sqrt.approx.f32 %0, %1;" : "=f"(r) : "f"(v));
  return r;
}

// One parameter: gradient g (l2 term included), slots s0 / s1 updated in place; returns the new value.
// Adam is the Keras form (eps outside the bias correction).  sqrt.approx / div.approx (<= 2 ulp each): the IEEE
// forms cost ~25 instructions per parameter, a fifth of the whole kernel at Dense32 sizes, for digits far below
// fp32 re-association noise.  The other kinds restate the training_ops.cc functors (RMSprop without momentum:
// the Python path of rmsprop.py) with the same approximate forms.
template <bool OPT>
__device__ __forceinline__ float opt_update(const OptHyper &h, const OptStep &s, float wv, float g, float &s0,
                                            float &s1) {
  if (OPT) {
    switch (h.kind) {
      case BORE_OPT_RMSPROP:
        if (h.momentum > 0.f) {  // ResourceApplyRMSProp: eps inside the root
          s0 += (g * g - s0) * s.om1;
          s1 = h.momentum * s1 + h.lr * g * rsqrtf(s0 + h.eps);
          return wv - s1;
        } else {
          s0 = h.b1 * s0 + s.om1 * (g * g);
          float den = s0;
          if (h.centered) {
            s1 = h.b1 * s1 + s.om1 * g;
            den = s0 - s1 * s1;
          }
          return wv - __fdividef(h.lr * g, sqrt_approx(den) + h.eps);
        }
      case BORE_OPT_ADAGRAD:  // ResourceApplyAdagradV2
        s0 += g * g;
        return wv - __fdividef(h.lr * g, sqrt_approx(s0) + h.eps);
      case BORE_OPT_ADADELTA: {  // ResourceApplyAdadelta
        s0 = s0 * h.b1 + (g * g) * s.om1;
        const float u = sqrt_approx(s1 + h.eps) * rsqrtf(s0 + h.eps) * g;
        s1 = s1 * h.b1 + (u * u) * s.om1;
        return wv - u * h.lr;
      }
      case BORE_OPT_ADAMAX:  // ResourceApplyAdaMax
        s0 += (g - s0) * s.om1;
        s1 = fmaxf(h.b2 * s1, fabsf(g));
        return wv - s.alpha * __fdividef(s0, s1 + h.eps);
      case BORE_OPT_NADAM: {  // nadam.py _resource_apply_dense
        s0 = h.b1 * s0 + s.om1 * g;
        s1 = h.b2 * s1 + s.om2 * (g * g);
        const float mbar = s.cg * g + s.cm * s0;
        return wv - __fdividef(h.lr * mbar, sqrt_approx(s1 * s.vd) + h.eps);
      }
      default: break;
    }
  }
  s0 += (g - s0) * s.om1;
  s1 += (g * g - s1) * s.om2;
  return wv - __fdividef(s0 * s.alpha, sqrt_approx(s1) + h.eps);
}

}  // namespace
