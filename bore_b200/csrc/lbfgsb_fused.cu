// K3f: the whole multi-start argmax in ONE persistent launch (sm_100a).
//
// Replaces the serial per-start loop of bore/mixins.py:57-61 -- scipy.optimize.minimize
// (L-BFGS-B) calling the value_and_gradient closure of bore/base.py:35-42 once per evaluation --
// with the same call chain per start, entirely on the device:
//
//     one WARP owns one start from x0 to termination.  Its L-BFGS-B state (lbfgsb_core.h,
//     the algorithm SciPy wraps) never leaves shared memory; whenever the state machine posts a
//     trial point the warp evaluates the MLP and its input gradient ITSELF (forward + reverse
//     through the input, FP32 FFMA, weights staged once per CTA in shared memory) and goes on.
//     A finished warp claims the next start from a global queue.
//
// What this removes compared with the lock-step round design of lbfgsb.cu (K2 launch + stepper
// launch per round, still used by the reverse-communication API for caller-supplied objectives):
// two launches per round (>= 300 rounds for 65,536 starts; a latency floor of ~93 us per round
// once few starts are active), the 14 KB per-start state streaming through HBM every round
// (0.94 GB for 65,536 starts of 50-D), the staging / write-back / list bookkeeping around every
// step (25 % of the stepper's instructions and 22 % of its stall samples in round 1,
// profiles/r01_notes.md), and the separate K2 launches with their input gather / gradient
// scatter through HBM.
//
// Two addressing modes, as in K2: all S starts belong to one model (the CTAs are persistent, one
// per SM, the warps pull starts from one queue), or start i belongs to model i / per_model
// (batched BO problems, BASELINE.json configs[3]): a CTA claims a MODEL, stages its weights,
// its warps run that model's starts, and it claims the next model.
//
// MLP evaluation by one warp.  Weights sit in shared memory in ONE layout, W[k][j], every layer
// padded to the net's width class (16 / 32 / 64 / 128 units) with leading dimension LD = width + 4:
// the forward pass walks rows (a lane owns width/32 adjacent output units: one LDS.32/64/128 per
// k, lanes contiguous), the reverse pass walks columns (a lane owns input unit k and reads
// W[k][j..j+3] as one LDS.128; LD / 4 is odd, so the 8 lanes of a quarter-warp hit 32 distinct
// banks) -- both directions conflict-free WITHOUT the transposed copy K2 keeps, which would cost
// the shared memory of two more resident starts.  The strides are compile-time constants (one
// instantiation per width class), so every load is [register + immediate].  Activations of the
// point live in a per-warp strip that aliases the K-matrix scratch of the optimiser (dead while
// the MLP runs).
#include <float.h>
#include <math.h>
#include <stdlib.h>

#include <algorithm>

#include "common.cuh"
#include "act.cuh"
#include "lbfgsb_fused.h"
#include "lbfgsb_types.h"

// The fused kernel is bound by instruction fetch (free-running warps, ~90 KB executed footprint):
// its copy of the core keeps the hot inner loops rolled (BORE: -DLB_FUSED_UNROLL restores unroll 2).
#ifndef LB_FUSED_UNROLL
#define LB_COMPACT 1
#endif
namespace lbf {  // warp-collective variant of the core, run-time history size m
#define LB_VARIANT 1
#include "lbfgsb_core.h"
#undef LB_VARIANT
}  // namespace lbf
namespace lbf10 {  // m = 10 (SciPy's default maxcor) as a compile-time constant
#define LB_VARIANT 1
#define LB_MCONST 10
#include "lbfgsb_core.h"
#undef LB_MCONST
#undef LB_VARIANT
}  // namespace lbf10

namespace {

template <int MC> struct Core;
template <> struct Core<0> {
  using Work = lbf::LbWork;
  template <class Mem>
  static __device__ __forceinline__ int advance(const LbParams &P, Work &w, LbScal &s, Mem &mem, int stage) {
    return lbf::lb_advance(P, w, s, mem, stage);
  }
  static __device__ __forceinline__ void init_state(const LbParams &P, Work &w, LbScal &s) {
    lbf::lb_init_state(P, w, s);
  }
  static __device__ __forceinline__ void prep_ld(Work &w, int m, int col) { lbf::lb_prep_ld(w, m, col); }
  using NoMem = lbf::LbNoMem;
};
template <> struct Core<10> {
  using Work = lbf10::LbWork;
  template <class Mem>
  static __device__ __forceinline__ int advance(const LbParams &P, Work &w, LbScal &s, Mem &mem, int stage) {
    return lbf10::lb_advance(P, w, s, mem, stage);
  }
  static __device__ __forceinline__ void init_state(const LbParams &P, Work &w, LbScal &s) {
    lbf10::lb_init_state(P, w, s);
  }
  static __device__ __forceinline__ void prep_ld(Work &w, int m, int col) { lbf10::lb_prep_ld(w, m, col); }
  using NoMem = lbf10::LbNoMem;
};

__host__ __device__ inline size_t f_align(size_t a, size_t b) { return (a + b - 1) / b * b; }
__host__ __device__ inline int f_rup(int a, int b) { return (a + b - 1) / b * b; }

// Shared-memory plan of the weight image and of one warp's activation strips (floats).
struct FusedPlan {
  int G;                          // hidden (GEMM) layers = n_layers - 1
  int D;                          // input dimension
  int width;                      // width class: 16, 32, 64 or 128 >= every hidden width
  int in[BORE_MAX_LAYERS];        // fan-in of layer l
  int out[BORE_MAX_LAYERS];       // fan-out
  int w[BORE_MAX_LAYERS];         // offset of W_l: rows = fan-in rounded up to 4, leading dim width + 4
  int b[BORE_MAX_LAYERS];         // offset of b_l (width entries)
  int act[BORE_MAX_LAYERS];       // activation of layer l (act[G] = the final Dense(1))
  int wl, wl_len;                 // final layer's weight vector, padded to a multiple of 4
  int total;                      // floats in the image
  int strip[BORE_MAX_LAYERS + 1]; // strip[0] = x, strip[l + 1] = output of layer l
  int strip_total;                // floats per warp
  int b_last;                     // offset of the final bias inside the flat parameter vector
};

void make_fused_plan(const MlpDesc &d, FusedPlan &p) {
  const int G = d.n_layers - 1;
  p.G = G;
  p.D = d.dims[0];
  int widest = 1;
  for (int l = 1; l <= G; ++l) widest = std::max(widest, d.dims[l]);
  p.width = widest <= 16 ? 16 : widest <= 32 ? 32 : widest <= 64 ? 64 : 128;
  const int LD = p.width + 4;
  int off = 0, so = 0;
  p.strip[0] = so; so += f_rup(d.dims[0], 4);
  for (int l = 0; l < G; ++l) {
    p.in[l] = d.dims[l]; p.out[l] = d.dims[l + 1];
    p.act[l] = d.act[l];
    p.w[l] = off; off += f_rup(d.dims[l], 4) * LD;
    p.b[l] = off; off += p.width;
    p.strip[l + 1] = so; so += p.width;
  }
  p.act[G] = d.act[G];
  p.wl_len = G > 0 ? p.width : f_rup(d.dims[0], 4);
  p.wl = off; off += p.wl_len;
  p.total = off;
  p.strip_total = so;
  p.b_last = d.b_off[G];
}

struct FusedArgs {
  LbParams P;                 // lo / hi / nbd: device pointers
  int S;                      // starts in total
  int per_model, n_models;    // per_model == 0: all starts belong to one model
  const double *X0;           // [S][n] start points
  double *x;                  // [S][n] final iterates
  double *fun;                // [S]
  int *nit, *nfev, *status, *task;  // [S] (each may be NULL)
  const float *params;        // flat Keras-order parameters of the first model
  int n_params;
  int transform;
  int nphase;                 // < 0: free-running warps; >= 0: CTA rendezvous before a heavy stage
  int *qhead;                 // queue head: next unclaimed start (one model) / model (batched)
  unsigned long long *evals;  // evaluations performed
  size_t warp_bytes;          // shared memory per warp
  // Resume mode (the tail of a lock-step run, lbfgsb.cu): instead of x0, a start comes with its
  // persisted state block and a pending request; results go back into the block.
  const int *resume_list;     // [*resume_count] start ids, or NULL
  const int *resume_count;
  char *blocks;               // persisted blocks (layout of lbfgsb_types.h), stride block_stride
  size_t block_stride;
  FusedPlan plan;
};

// CTA header in dynamic shared memory
struct FusedHeader {
  FusedPlan plan;
  int transform;
  int unit;       // batched mode: the model this CTA works on
  float b_last;
};
__host__ __device__ inline size_t fused_header_bytes(int n) {
  return f_align(LB_FORMK_ACC * 32 * sizeof(int), 16) + 2 * f_align(n * sizeof(double), 16) +
         f_align(n * sizeof(int), 16) + f_align(sizeof(FusedHeader), 16);
}

// T adjacent floats from shared memory as one load
template <int T> struct FVec;
template <> struct FVec<1> { float v[1]; __device__ __forceinline__ void load(const float *p) { v[0] = *p; }
                             __device__ __forceinline__ void store(float *p) const { *p = v[0]; } };
template <> struct FVec<2> { float v[2]; __device__ __forceinline__ void load(const float *p) {
                               const float2 t = *reinterpret_cast<const float2 *>(p); v[0] = t.x; v[1] = t.y; }
                             __device__ __forceinline__ void store(float *p) const {
                               *reinterpret_cast<float2 *>(p) = make_float2(v[0], v[1]); } };
template <> struct FVec<4> { float v[4]; __device__ __forceinline__ void load(const float *p) {
                               const float4 t = *reinterpret_cast<const float4 *>(p);
                               v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w; }
                             __device__ __forceinline__ void store(float *p) const {
                               *reinterpret_cast<float4 *>(p) = make_float4(v[0], v[1], v[2], v[3]); } };

// One warp: f = T(-u(x)), g = df/dx for the point in x[0..D) (fp64 in, fp32 arithmetic, fp64 out
// -- the dtype flow of bore/decorators.py:54-56).  `strip` is the warp's activation scratch.
// WIDTH = the net's width class; a lane owns T = WIDTH / 32 (>= 1) adjacent output units on the
// way forward and input units lane, lane + 32, ... on the way back.
template <int WIDTH, bool EXT>
__device__ __noinline__ float fused_eval(const FusedHeader *H, const float *__restrict__ wsm,
                                         float *__restrict__ strip, const double *__restrict__ x,
                                         double *__restrict__ g) {
  __builtin_assume(__isShared(H)); __builtin_assume(__isShared(wsm));
  __builtin_assume(__isShared(strip)); __builtin_assume(__isShared(x)); __builtin_assume(__isShared(g));
  constexpr int LD = WIDTH + 4;
  constexpr int T = WIDTH >= 32 ? WIDTH / 32 : 1;
  const FusedPlan &pl = H->plan;
  const int lane = threadIdx.x & 31;
  const int G = pl.G;
  const int D = pl.D;
  {
    // fp32 copy of the point; the pad up to a multiple of 4 is written as zeros
    float *x0 = strip + pl.strip[0];
    const int D4 = f_rup(D, 4);
#pragma unroll 1
    for (int k = lane; k < D4; k += 32) x0[k] = k < D ? (float)x[k] : 0.f;
  }
  __syncwarp();
  // ---- forward through the hidden layers ----
  const int j0 = T * lane;
#pragma unroll 1
  for (int l = 0; l < G; ++l) {
    const int in4 = f_rup(pl.in[l], 4), a = pl.act[l];
    const float *A = strip + pl.strip[l];
    float *Hn = strip + pl.strip[l + 1];
    if (j0 < WIDTH) {
      const float *W = wsm + pl.w[l] + j0;
      // ONE accumulator per output, k ascending: the summation order of K2's tile_gemm, so that
      // this evaluation is bit-identical to mlp_eval_kernel's (a start may change hands between the
      // two in mid line search, lbfgsb.cu; mixed roundings would bias its sufficient-decrease tests)
      float acc[T];
#pragma unroll
      for (int t = 0; t < T; ++t) acc[t] = 0.f;
#pragma unroll 2
      for (int k = 0; k < in4; k += 4) {
        const float4 x4 = *reinterpret_cast<const float4 *>(A + k);
        FVec<T> w0, w1, w2, w3;
        w0.load(W); w1.load(W + LD); w2.load(W + 2 * LD); w3.load(W + 3 * LD);
        W += 4 * LD;
#pragma unroll
        for (int t = 0; t < T; ++t) {
          acc[t] = fmaf(x4.x, w0.v[t], acc[t]);
          acc[t] = fmaf(x4.y, w1.v[t], acc[t]);
          acc[t] = fmaf(x4.z, w2.v[t], acc[t]);
          acc[t] = fmaf(x4.w, w3.v[t], acc[t]);
        }
      }
      FVec<T> bv, hv;
      bv.load(wsm + pl.b[l] + j0);
#pragma unroll
      for (int t = 0; t < T; ++t) hv.v[t] = act_fwd<EXT>(a, acc[t] + bv.v[t]);
      hv.store(Hn + j0);  // pad units: zero weights and bias -> act(0), multiplied by zero rows later
    }
    __syncwarp();
  }
  // ---- final Dense(1) ----
  float *HL = strip + pl.strip[G];
  const float *wl = wsm + pl.wl;
  // (K2's association: UG = 16 (8 for nets no wider than 32) partial sums over k = ug, ug + UG, ...,
  // combined by an xor butterfly; both half-warps compute the same value)
  float up = 0.f;
  {
    const int UG = WIDTH > 32 ? 16 : 8;
#pragma unroll 1
    for (int k = lane & (UG - 1); k < pl.wl_len; k += UG) up = fmaf(HL[k], wl[k], up);  // (pad terms are +0)
#pragma unroll
    for (int o = 1; o < UG; o <<= 1) up += __shfl_xor_sync(0xffffffffu, up, o);
  }
  const int act_last = pl.act[G];
  const float u = act_fwd<EXT>(act_last, up + H->b_last);
  const float v = -u;  // the mixin minimises transform(-u) (bore/mixins.py:20)
  float fval, dT;
  if (H->transform == BORE_TRANSFORM_SIGMOID) {
    fval = 1.f / (1.f + expf(-v));
    dT = fval * (1.f - fval);
  } else if (H->transform == BORE_TRANSFORM_EXP) {
    fval = expf(v);
    dT = fval;
  } else {
    fval = v;
    dT = 1.f;
  }
  const float dpre = -dT * act_bwd<EXT>(act_last, u);
  // ---- reverse through the input ----
  if (G == 0) {
#pragma unroll 1
    for (int k = lane; k < D; k += 32) g[k] = (double)(dpre * wl[k]);
    __syncwarp();
    return fval;
  }
  {
    const int a = pl.act[G - 1];
#pragma unroll 1
    for (int k = lane; k < WIDTH; k += 32) HL[k] = dpre * wl[k] * act_bwd<EXT>(a, HL[k]);  // (wl pad is zero)
  }
  __syncwarp();
#pragma unroll 1
  for (int l = G - 1; l >= 0; --l) {
    const int in = pl.in[l], out4 = f_rup(pl.out[l], 4);
    const float *Dl = strip + pl.strip[l + 1];  // delta of the layer's output
    float *Hin = strip + pl.strip[l];
    const float *W = wsm + pl.w[l];
    const int a = l > 0 ? pl.act[l - 1] : 0;
#pragma unroll 1
    for (int i0 = 0; i0 < in; i0 += 64) {
      const int ia = i0 + lane, ib = ia + 32;
      const bool va = ia < in, vb = ib < in;
      const bool two = i0 + 32 < in;  // (warp-uniform) the second row block exists
      const float *ra = W + (va ? ia : 0) * LD, *rb = W + (vb ? ib : 0) * LD;
      float a0 = 0.f, b0 = 0.f;  // one accumulator per unit, j ascending (K2's order)
      if (two) {
#pragma unroll 2
        for (int j = 0; j < out4; j += 4) {
          const float4 d4 = *reinterpret_cast<const float4 *>(Dl + j);
          const float4 wa = *reinterpret_cast<const float4 *>(ra + j);
          const float4 wb = *reinterpret_cast<const float4 *>(rb + j);
          a0 = fmaf(d4.x, wa.x, a0); b0 = fmaf(d4.x, wb.x, b0);
          a0 = fmaf(d4.y, wa.y, a0); b0 = fmaf(d4.y, wb.y, b0);
          a0 = fmaf(d4.z, wa.z, a0); b0 = fmaf(d4.z, wb.z, b0);
          a0 = fmaf(d4.w, wa.w, a0); b0 = fmaf(d4.w, wb.w, b0);
        }
      } else {
#pragma unroll 2
        for (int j = 0; j < out4; j += 4) {
          const float4 d4 = *reinterpret_cast<const float4 *>(Dl + j);
          const float4 wa = *reinterpret_cast<const float4 *>(ra + j);
          a0 = fmaf(d4.x, wa.x, a0);
          a0 = fmaf(d4.y, wa.y, a0);
          a0 = fmaf(d4.z, wa.z, a0);
          a0 = fmaf(d4.w, wa.w, a0);
        }
      }
      if (l > 0) {
        // in place: every lane reads and writes only its own units, the j loop reads the strip above
        if (va) Hin[ia] = a0 * act_bwd<EXT>(a, Hin[ia]);
        if (vb) Hin[ib] = b0 * act_bwd<EXT>(a, Hin[ib]);
      } else {
        if (va) g[ia] = (double)a0;
        if (vb) g[ib] = (double)b0;
      }
    }
    __syncwarp();
  }
  return fval;
}

template <bool EXT>
__device__ __forceinline__ float fused_eval_any(const FusedHeader *H, const float *wsm, float *strip,
                                                const double *x, double *g) {
  switch (H->plan.width) {  // warp-uniform
    case 16: return fused_eval<16, EXT>(H, wsm, strip, x, g);
    case 32: return fused_eval<32, EXT>(H, wsm, strip, x, g);
    case 64: return fused_eval<64, EXT>(H, wsm, strip, x, g);
    default: return fused_eval<128, EXT>(H, wsm, strip, x, g);
  }
}

// per-warp workspace: doubles, then ints (see carve below).  The MLP's activation strips alias
// the FIRST half of the K-matrix scratch wn (rows 0..m-1: formt / formk scratch, dead while the
// MLP runs) and, if they are larger, extra space in front of it; the second half holds ld.
__host__ __device__ inline size_t fused_strip_doubles(int m, int strip_floats) {
  const size_t half = 2 * (size_t)m * m;
  const size_t st = (((size_t)strip_floats + 1) / 2 + 1) & ~(size_t)1;
  return st > half ? st : half;  // doubles from the start of the strips to the middle of wn
}
__host__ __device__ inline size_t fused_warp_bytes(int n, int m, int strip_floats) {
  const size_t nv = LB_NV(n);
  const size_t d = 6 * nv + LB_NW(n, m) + ((4 * (size_t)m * m + 1) & ~(size_t)1) +
                   fused_strip_doubles(m, strip_floats) + 2 * (size_t)m * m + 12 * (size_t)m;
  return f_align(d * sizeof(double) + 2 * (size_t)n * sizeof(int), 16);
}

template <class Work>
__device__ __forceinline__ float *fused_carve(Work &w, unsigned char *base, int n, int m, int strip_floats) {
  double *q = reinterpret_cast<double *>(base);
  const int nv = LB_NV(n);
  w.x = q; q += nv; w.g = q; q += nv; w.t = q; q += nv; w.r = q; q += nv; w.d = q; q += nv; w.z = q; q += nv;
  w.xp = w.t;  // the Cauchy breakpoints (t) are dead when subsm saves the Cauchy point
  w.W = q; q += LB_NW(n, m);
  w.sy = q; q += m * m; w.ss = q; q += m * m; w.yy = q; q += m * m; w.tinv = q; q += m * m;
  if ((4 * m * m) & 1) ++q;  // the scratch starts 16-byte aligned (float4 loads of the strips)
  float *strip = reinterpret_cast<float *>(q);
  q += fused_strip_doubles(m, strip_floats);  // -> the middle of wn
  w.wn = q - 2 * m * m;
  w.ld = q;                                   // == w.wn + m * LB_LDL(m)
  q += 2 * m * m;
  w.rd = q; q += 2 * m;
  w.p = q; q += 2 * m; w.c = q; q += 2 * m; w.wbp = q; q += 2 * m; w.v = q; q += 2 * m; w.q = q; q += 2 * m;
  int *ib = reinterpret_cast<int *>(q);
  w.iwhere = ib; w.index = ib + n;
  w.ftab = nullptr;
  w.changed = 0;
  return strip;
}

constexpr int FUSED_MAX_WARPS = 12;

template <int MC, bool EXT>
__global__ void __launch_bounds__(FUSED_MAX_WARPS * 32, 1) lbfgsb_fused_kernel(const FusedArgs A) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int n = A.P.n, m = MC ? MC : A.P.m;
  const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  const bool multi = A.per_model > 0;
  const bool aligned = A.nphase >= 0;
  const bool strict = A.nphase >= 1;

  // ---- CTA header ----
  unsigned char *sp = smem_raw;
  int *ftab = reinterpret_cast<int *>(sp); sp += f_align(LB_FORMK_ACC * 32 * sizeof(int), 16);
  double *s_lo = reinterpret_cast<double *>(sp); sp += f_align(n * sizeof(double), 16);
  double *s_hi = reinterpret_cast<double *>(sp); sp += f_align(n * sizeof(double), 16);
  int *s_nbd = reinterpret_cast<int *>(sp); sp += f_align(n * sizeof(int), 16);
  FusedHeader *H = reinterpret_cast<FusedHeader *>(sp); sp += f_align(sizeof(FusedHeader), 16);
  float *wsm = reinterpret_cast<float *>(sp); sp += f_align((size_t)A.plan.total * sizeof(float), 16);
  unsigned char *wbase = sp + A.warp_bytes * wib;

#pragma unroll 1
  for (int o = threadIdx.x; o < LB_FORMK_ACC * 32; o += blockDim.x) ftab[o] = lbf::lb_formk_code(o, m);
#pragma unroll 1
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    s_lo[i] = A.P.lo[i];
    s_hi[i] = A.P.hi[i];
    s_nbd[i] = A.P.nbd[i];
  }
  if (threadIdx.x == 0) {
    H->plan = A.plan;
    H->transform = A.transform;
    H->unit = 0;
  }
  LbParams P = A.P;
  P.lo = s_lo; P.hi = s_hi; P.nbd = s_nbd;

  typename Core<MC>::Work w;
  float *strip = fused_carve(w, wbase, n, m, A.plan.strip_total);
  w.ftab = ftab;
  typename Core<MC>::NoMem mem;
  LbScal s;
  unsigned long long my_evals = 0;
  const FusedPlan &pl = A.plan;

#pragma unroll 1
  for (;;) {  // units: the one model, or one model after the other
    int model = 0;
    if (multi) {
      if (threadIdx.x == 0) H->unit = atomicAdd(A.qhead, 1);
      __syncthreads();  // (every warp is done with the previous model's weights)
      model = H->unit;
      if (model >= A.n_models) break;
    }
    // ---- stage this model's weights: W_l [k][j] with an odd leading dimension, zero padded ----
    {
      const float *params = A.params + (size_t)model * A.n_params;
#pragma unroll 1
      for (int e = threadIdx.x; e < pl.total; e += blockDim.x) wsm[e] = 0.f;
      __syncthreads();
      // (the flat parameter vector is [W_0 b_0 W_1 b_1 ...]; offsets recomputed here)
      int off = 0;
      const int LD = pl.width + 4;
#pragma unroll 1
      for (int l = 0; l < pl.G; ++l) {
        const int in = pl.in[l], out = pl.out[l];
        float *Wd = wsm + pl.w[l];
#pragma unroll 1
        for (int k = wib; k < in; k += wpb)
#pragma unroll 1
          for (int j = lane; j < out; j += 32) Wd[k * LD + j] = params[off + k * out + j];
        off += in * out;
        float *Bd = wsm + pl.b[l];
#pragma unroll 1
        for (int e = threadIdx.x; e < out; e += blockDim.x) Bd[e] = params[off + e];
        off += out;
      }
      const int inl = pl.G > 0 ? pl.out[pl.G - 1] : n;
#pragma unroll 1
      for (int e = threadIdx.x; e < inl; e += blockDim.x) wsm[pl.wl + e] = params[off + e];
      if (threadIdx.x == 0) H->b_last = params[pl.b_last];
    }
    __syncthreads();

    int k_local = wib;  // batched mode: this warp's next start of the model
    const int n_items = A.resume_list ? *A.resume_count : A.S;
    bool resumed_first = false;
    int sid = -1;
    bool have = false;
    int stage = aligned ? 1 : 0;
#pragma unroll 1
    for (;;) {
      bool fresh = false;
      const bool was_heavy = stage == 2;
      if (stage != 2 && !have) {
        // ---- claim a start ----
        if (multi) {
          sid = k_local < A.per_model ? model * A.per_model + k_local : -1;
          k_local += wpb;
        } else {
          int v = 0;
          if (lane == 0) v = atomicAdd(A.qhead, 1);
          v = __shfl_sync(0xffffffffu, v, 0);
          sid = v < n_items ? v : -1;
        }
        if (sid >= 0 && A.resume_list) {
          // ---- resume: the start's persisted block (scalars | t r d z | W | sy ss yy tinv) and
          //      its pending request; the evaluation that follows was counted when it was posted
          sid = A.resume_list[sid];
          const double *blk = reinterpret_cast<const double *>(A.blocks + A.block_stride * sid);
          s = *reinterpret_cast<const LbScal *>(blk);
          const double *src = blk + LB_SCAL_DOUBLES;
          const int nv = LB_NV(n);
#pragma unroll 1
          for (int i = lane; i < n; i += 32) {
            w.t[i] = src[i]; w.r[i] = src[nv + i]; w.d[i] = src[2 * nv + i]; w.z[i] = src[3 * nv + i];
            w.x[i] = A.x[(size_t)sid * n + i];
            const int nb = s_nbd[i];
            w.iwhere[i] = nb == 0 ? -1 : ((nb == 2 && s_hi[i] - s_lo[i] <= 0.0) ? 3 : 0);
          }
          src += 4 * nv;
          const int nmat = LB_NW(n, m) + 4 * m * m;  // W and the four matrices are contiguous on both sides
#pragma unroll 1
          for (int i = lane; i < nmat; i += 32) w.W[i] = src[i];
          __syncwarp();
          if (s.col > 0) Core<MC>::prep_ld(w, m, s.col);
          have = true;
          fresh = true;
          resumed_first = true;
        } else if (sid >= 0) {
          const double *x0 = A.X0 + (size_t)sid * n;
#pragma unroll 1
          for (int i = lane; i < n; i += 32) w.x[i] = x0[i];
          __syncwarp();
          Core<MC>::init_state(P, w, s);  // clips x0 into the box like SciPy (_lbfgsb_py.py:359)
          s.nfev = 1;                     // the evaluation at x0
          have = true;
          fresh = true;
        }
      }
      bool arrive = !have, holding = false;
      if (have) {
        int r = 1;
        if (!fresh) {
          r = Core<MC>::advance(P, w, s, mem, stage);  // the only call site of the state machine
          if (r == 1 && w.changed) s.nfev += 1;
        }
        if (r == 2) {
          holding = true;
          arrive = true;
        } else {
          if (stage == 2) stage = 1;
          if (r == 1) {
            s.f = (double)fused_eval_any<EXT>(H, wsm, strip, w.x, w.g);
            if (!resumed_first) my_evals += 1;
            resumed_first = false;
          } else {
            // ---- terminated: final iterate and counters ----
            double *xo = A.x + (size_t)sid * n;
#pragma unroll 1
            for (int i = lane; i < n; i += 32) xo[i] = w.x[i];
            if (lane == 0 && A.resume_list)
              *reinterpret_cast<LbScal *>(A.blocks + A.block_stride * sid) = s;  // read by the results kernel
            if (lane == 0) {
              if (A.fun) A.fun[sid] = s.f;
              if (A.nit) A.nit[sid] = s.nit;
              if (A.nfev) A.nfev[sid] = s.nfev;
              if (A.status) A.status[sid] = s.status;
              if (A.task) A.task[sid] = s.task;
            }
            have = false;
          }
        }
      }
      if (!aligned) {
        if (!have && sid < 0) break;
        continue;
      }
      if (strict) {
        // lock-step rounds inside the persistent kernel: [light stage (+ evaluation) of every warp]
        // barrier [heavy stage (+ evaluation) of the warps that begin a new iteration] barrier
        if (!was_heavy) {
          __syncthreads_or(0);
          if (holding) { stage = 2; continue; }
        }
        const int alive = __syncthreads_or((have || sid >= 0) ? 1 : 0);
        if (!alive) break;
        stage = 1;
        continue;
      }
      if (arrive) {
        if (!__syncthreads_or(holding ? 1 : 0)) break;  // nobody holds an item and nobody has work
        stage = holding ? 2 : 1;
      }
    }
    if (!multi) break;
  }
  if (lane == 0 && my_evals) atomicAdd(A.evals, my_evals);
}

template <int MC, bool EXT>
int launch_fused_mc(const FusedArgs &A, int grid, int block, size_t smem, cudaStream_t stream) {
  static bool attr_done[64] = {};
  int dev = 0;
  BORE_CUDA(cudaGetDevice(&dev));
  if (dev >= 64 || !attr_done[dev]) {
    BORE_CUDA(cudaFuncSetAttribute(lbfgsb_fused_kernel<MC, EXT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   227 * 1024));
    if (dev < 64) attr_done[dev] = true;
  }
  lbfgsb_fused_kernel<MC, EXT><<<grid, block, smem, stream>>>(A);
  BORE_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace

// ---------------------------------------------------------------- host side
size_t lbfgsb_fused_workspace_bytes(int n) {
  return 64 + 2 * f_align(n * sizeof(double), 16) + f_align(n * sizeof(int), 16);
}

// 1 when the fused kernel can run this problem (weights + at least `min_warps` resident starts fit
// into one SM's shared memory), else 0: the caller then uses the lock-step round path.
int lbfgsb_fused_fits(const bore_mlp *h, int m) {
  FusedPlan pl;
  make_fused_plan(h->desc, pl);
  const int n = h->desc.dims[0];
  const size_t need = fused_header_bytes(n) + f_align((size_t)pl.total * sizeof(float), 16) +
                      2 * fused_warp_bytes(n, m, pl.strip_total);
  return need <= (size_t)227 * 1024 ? 1 : 0;
}

int launch_lbfgsb_fused(const bore_mlp *h, int model0, int n_models, int per_model, int transform,
                        const double *X0_dev, int S, const LbParams &P_dev, void *work_dev,
                        double *x_dev, double *fun_dev, int *nit_dev, int *nfev_dev, int *status_dev,
                        int *task_dev, long long *evals_out, FusedLaunchInfo *info, cudaStream_t stream,
                        const FusedResume *resume) {
  const int n = h->desc.dims[0], m = P_dev.m;
  FusedArgs A;
  make_fused_plan(h->desc, A.plan);
  A.P = P_dev;
  A.S = S;
  A.per_model = per_model;
  A.n_models = n_models;
  A.X0 = X0_dev;
  A.x = x_dev; A.fun = fun_dev; A.nit = nit_dev; A.nfev = nfev_dev; A.status = status_dev; A.task = task_dev;
  A.params = h->params + (size_t)model0 * h->desc.n_params;
  A.n_params = h->desc.n_params;
  A.transform = transform;
  {
    static int nphase = -2;
    if (nphase == -2) {
      const char *e = getenv("BORE_LBF_NPHASE");
      nphase = e ? atoi(e) : -1;
      if (nphase < -1) nphase = -1;
    }
    A.nphase = nphase;
  }
  A.qhead = reinterpret_cast<int *>(work_dev);
  A.evals = reinterpret_cast<unsigned long long *>(static_cast<char *>(work_dev) + 8);
  A.resume_list = nullptr; A.resume_count = nullptr; A.blocks = nullptr; A.block_stride = 0;
  if (resume) {
    // S = an upper bound of the number of starts still running; the kernel reads the exact count
    A.resume_list = resume->list; A.resume_count = resume->count;
    A.blocks = resume->blocks; A.block_stride = resume->block_stride;
    A.qhead = resume->qhead; A.evals = resume->evals;
  }
  A.warp_bytes = fused_warp_bytes(n, m, A.plan.strip_total);
  const size_t fixed = fused_header_bytes(n) + f_align((size_t)A.plan.total * sizeof(float), 16);
  const size_t max_block = 227 * 1024, max_sm = 228 * 1024;
  BORE_CHECK(fixed + A.warp_bytes <= max_block, "lbfgsb (fused): model + one start need %zu B of shared memory",
             fixed + A.warp_bytes);
  int wmax = (int)((max_block - fixed) / A.warp_bytes);
  if (wmax > FUSED_MAX_WARPS) wmax = FUSED_MAX_WARPS;
  {
    static int forced = -1;
    if (forced < 0) {
      const char *e = getenv("BORE_LBF_WPB");
      forced = e ? atoi(e) : 0;
    }
    if (forced >= 1 && forced <= wmax) wmax = forced;
  }
  int wpb, grid;
  if (per_model > 0) {
    wpb = std::min(per_model, wmax);
    int per_sm = (int)(max_sm / (fixed + wpb * A.warp_bytes + 1024));
    if (per_sm * wpb > FUSED_MAX_WARPS) per_sm = FUSED_MAX_WARPS / wpb;
    if (per_sm < 1) per_sm = 1;
    grid = std::min(n_models, h->sm_count * per_sm);
  } else {
    // spread the starts over all SMs before stacking warps on one
    wpb = std::min(wmax, std::max(1, (S + h->sm_count - 1) / h->sm_count));
    grid = std::min(h->sm_count, (S + wpb - 1) / wpb);
  }
  const size_t smem = fixed + wpb * A.warp_bytes;
  if (resume) BORE_CUDA(cudaMemsetAsync(resume->qhead, 0, sizeof(int), stream));
  else BORE_CUDA(cudaMemsetAsync(work_dev, 0, 16, stream));
  const bool ext = acts_ext(h->desc.act, h->desc.n_layers);
  const int rc = m == 10 ? (ext ? launch_fused_mc<10, true>(A, grid, wpb * 32, smem, stream)
                                : launch_fused_mc<10, false>(A, grid, wpb * 32, smem, stream))
                         : (ext ? launch_fused_mc<0, true>(A, grid, wpb * 32, smem, stream)
                                : launch_fused_mc<0, false>(A, grid, wpb * 32, smem, stream));
  if (rc) return rc;
  if (info) { info->grid = grid; info->block = wpb * 32; info->smem = smem; }
  if (evals_out) {
    unsigned long long ev = 0;
    BORE_CUDA(cudaMemcpyAsync(&ev, A.evals, sizeof(ev), cudaMemcpyDeviceToHost, stream));
    BORE_CUDA(cudaStreamSynchronize(stream));
    *evals_out = (long long)ev;
  }
  return 0;
}
