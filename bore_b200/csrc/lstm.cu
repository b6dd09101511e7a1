// K7: the LSTM multi-fidelity classifier of the reference (SURVEY.md section 8f, row 4) on sm_100a.
//
// Replaces the Keras networks StackedRecurrentFactory builds (bore/models.py:48-104):
//   many-to-many   Masking -> RNN(LSTMCell, return_sequences=True) x L -> TimeDistributed(Dense(1)),
//                  trained by fit() on sequences padded with mask_value
//                  (bore/plugins/hpbandster/multi_fidelity.py:198-233, bore/data.py:183-251);
//   one-to-one     RepeatVector(num_steps) -> the same cells -> the same Dense on the last step,
//                  the MaximizableSequential whose argmax proposes the next configuration
//                  (multi_fidelity.py:262-278) -- value and input gradient for the L-BFGS-B stepper.
//
// Mapping.  The model is tiny (U <= 32 units, L <= 4 cells, T <= 8 rungs) and every sample is an
// independent recurrence: ONE WARP carries one sample through all steps and layers, lane = unit.
// The weights of a cell sit in shared memory as one matrix [x ; h] -> 4U gates with an ODD leading
// dimension (4U + 1): the forward pass reads rows (lane = gate column: consecutive words), the
// reverse pass reads columns (lane = input row: stride 4U + 1 -> 32 distinct banks).  Per step and
// cell a lane keeps i, f, c~, o, act(c) and c_prev of its unit in the warp's shared-memory strip for
// the way back (BPTT).  Masked steps (all features == mask_value) carry state and output through,
// as keras.backend.rnn does.
//
// Training (lstm_fit_kernel): the whole fit in one launch, one CTA; per Adam step the warps run
// forward + BPTT for the samples of the minibatch and leave, per (cell, step, sample), the input row
// [x ; h_prev] and the gate gradient dz in an L2-resident scratch; the weight gradients are then
// small GEMMs  dW = sum_b [x ; h_prev]_b' dz_b  (staged through shared memory, 32 outputs per
// thread), followed by the Keras-form Adam update in place.  Deterministic (no atomics).
#include <algorithm>

#include "common.cuh"
#include "act.cuh"
#include "opt.cuh"

#define LSTM_MAX_LAYERS 4
#define LSTM_MAX_UNITS 32
#define LSTM_MAX_DIM 32
#define LSTM_MAX_STEPS 8
#define LSTM_MAX_BATCH 64

struct LstmDesc {
  int D, U, L, act;
  int k_off[LSTM_MAX_LAYERS], r_off[LSTM_MAX_LAYERS], b_off[LSTM_MAX_LAYERS];  // flat Keras order
  int wd_off, bd_off, n_params;
  // shared-memory image: per cell Wcat [(in + U)][4U + 1] then bias [4U]; then wd [U], bd
  int s_w[LSTM_MAX_LAYERS], s_b[LSTM_MAX_LAYERS], s_wd, s_bd, s_total;
};

struct bore_lstm {
  LstmDesc desc;
  int device, sm_count;
  float *params, *adam_m, *adam_v;
  long long adam_t;
  float *opt_cache;  // (device, 1 float) Nadam's momentum cache
  OptHyper opt;
  LrSchedule sched;
  float l2[3 * LSTM_MAX_LAYERS + 2];  // per array, Keras order
  float l1[3 * LSTM_MAX_LAYERS + 2];
  float *scratch;
  size_t scratch_bytes;
};

namespace {

__device__ __forceinline__ float l_sigmoid(float v) { return 1.f / (1.f + expf(-v)); }

__host__ __device__ inline int in_dim(const LstmDesc &d, int l) { return l == 0 ? d.D : d.U; }
__host__ __device__ inline int ldw(const LstmDesc &d) { return 4 * d.U + 1; }

// stage the weight image of the model from its flat parameter vector (all threads of the CTA)
__device__ void stage_weights(const LstmDesc &d, const float *__restrict__ p, float *__restrict__ ws) {
  const int U = d.U, G4 = 4 * d.U, LD = ldw(d);
  for (int l = 0; l < d.L; ++l) {
    const int in = in_dim(d, l);
    float *W = ws + d.s_w[l];
    for (int e = threadIdx.x; e < (in + U) * G4; e += blockDim.x) {
      const int k = e / G4, j = e - k * G4;
      W[k * LD + j] = k < in ? p[d.k_off[l] + k * G4 + j] : p[d.r_off[l] + (k - in) * G4 + j];
    }
    for (int e = threadIdx.x; e < G4; e += blockDim.x) ws[d.s_b[l] + e] = p[d.b_off[l] + e];
  }
  for (int e = threadIdx.x; e < U; e += blockDim.x) ws[d.s_wd + e] = p[d.wd_off + e];
  if (threadIdx.x == 0) ws[d.s_bd] = p[d.bd_off];
}

// per-warp strip (floats): xin [D] | h [L][U] | c (registers) | dz [4U] | din [in_max + U] | acts [T][L][6][U]
__host__ __device__ inline int strip_floats(const LstmDesc &d, int T, bool keep) {
  const int inmax = d.D > d.U ? d.D : d.U;
  return ((d.D + d.L * d.U + 4 * d.U + inmax + d.U + (keep ? T * d.L * 6 * d.U : 0)) + 3) & ~3;
}
struct Strip {
  float *xin, *h, *dz, *din, *acts;
};
__device__ __forceinline__ Strip carve_strip(const LstmDesc &d, float *base) {
  Strip s;
  const int inmax = d.D > d.U ? d.D : d.U;
  s.xin = base; base += d.D;
  s.h = base; base += d.L * d.U;
  s.dz = base; base += 4 * d.U;
  s.din = base; base += inmax + d.U;
  s.acts = base;
  return s;
}

// One warp, one sample: the stack at step t.  h/c of every cell are updated in place (h in the
// strip, c in the caller's registers: c[l] is the state of unit `lane`).  With `keep` the gate
// values are stored for the way back.  `live` = the step is not masked.  Returns nothing; the top
// cell's output is s.h + (L-1)*U.
template <bool EXT>
__device__ __forceinline__ void stack_forward(const LstmDesc &d, const float *__restrict__ ws, const Strip &s,
                                              float (&c)[LSTM_MAX_LAYERS], int t, bool live, bool keep,
                                              int lane) {
  if (!live) return;  // states carried over, output = previous output (keras.backend.rnn, mask branch)
  const int U = d.U, LD = ldw(d), act = d.act;
  const bool on = lane < U;
  const int col = on ? lane : 0;
#pragma unroll 1
  for (int l = 0; l < d.L; ++l) {
    const int in = in_dim(d, l);
    const float *W = ws + d.s_w[l] + col;
    const float *bias = ws + d.s_b[l] + col;
    const float *xin = l == 0 ? s.xin : s.h + (l - 1) * U;
    float *hl = s.h + l * U;
    float z0 = bias[0], z1 = bias[U], z2 = bias[2 * U], z3 = bias[3 * U];
#pragma unroll 2
    for (int k = 0; k < in; ++k) {
      const float xv = xin[k];
      const float *w = W + k * LD;
      z0 = fmaf(xv, w[0], z0); z1 = fmaf(xv, w[U], z1); z2 = fmaf(xv, w[2 * U], z2); z3 = fmaf(xv, w[3 * U], z3);
    }
#pragma unroll 2
    for (int k = 0; k < U; ++k) {
      const float hv = hl[k];
      const float *w = W + (in + k) * LD;
      z0 = fmaf(hv, w[0], z0); z1 = fmaf(hv, w[U], z1); z2 = fmaf(hv, w[2 * U], z2); z3 = fmaf(hv, w[3 * U], z3);
    }
    const float gi = l_sigmoid(z0), gf = l_sigmoid(z1), gg = act_fwd<EXT>(act, z2), go = l_sigmoid(z3);
    const float cp = c[l];
    const float cn = gf * cp + gi * gg;
    const float ac = act_fwd<EXT>(act, cn);
    __syncwarp();  // every lane has read the old h of this cell
    if (on) {
      hl[lane] = go * ac;
      c[l] = cn;
      if (keep) {
        float *a = s.acts + ((size_t)(t * d.L + l) * 6) * U + lane;
        a[0] = gi; a[U] = gf; a[2 * U] = gg; a[3 * U] = go; a[4 * U] = ac; a[5 * U] = cp;
      }
    }
    __syncwarp();
  }
}

// One warp, one sample, ONE cell, one step back.  dht = total gradient wrt the cell's output h_t
// (from step t+1, from the layer above at this step, from the Dense layer), dc_in = gradient wrt
// c_t from step t+1.  Leaves the gate gradient dz (4U) in s.dz and  din = dz W'  (gradient wrt the
// cell's input, rows [0, in), and wrt h_{t-1}, rows [in, in+U)) in s.din; returns the gradient wrt
// c_{t-1} of unit `lane`.
template <bool EXT>
__device__ __forceinline__ float cell_backward(const LstmDesc &d, const float *__restrict__ ws, const Strip &s,
                                               int t, int l, float dht, float dc_in, int lane) {
  const int U = d.U, LD = ldw(d), act = d.act, G4 = 4 * U;
  const bool on = lane < U;
  const int in = in_dim(d, l);
  const float *a = s.acts + ((size_t)(t * d.L + l) * 6) * U + (on ? lane : 0);
  const float gi = a[0], gf = a[U], gg = a[2 * U], go = a[3 * U], ac = a[4 * U], cp = a[5 * U];
  const float d_o = dht * ac * go * (1.f - go);
  const float dct = dht * go * act_bwd<EXT>(act, ac) + dc_in;
  const float d_i = dct * gg * gi * (1.f - gi);
  const float d_f = dct * cp * gf * (1.f - gf);
  const float d_g = dct * gi * act_bwd<EXT>(act, gg);
  __syncwarp();
  if (on) { s.dz[lane] = d_i; s.dz[U + lane] = d_f; s.dz[2 * U + lane] = d_g; s.dz[3 * U + lane] = d_o; }
  __syncwarp();
  // din[k] = sum_j dz[j] W[k][j], k < in + U <= 64: lane = row (stride 4U + 1: conflict-free)
  float acc0 = 0.f, acc1 = 0.f;
  const int nr = in + U, r0 = lane, r1 = lane + 32;
  const float *W = ws + d.s_w[l];
  const float *w0 = W + (r0 < nr ? r0 : 0) * LD, *w1 = W + (r1 < nr ? r1 : 0) * LD;
#pragma unroll 2
  for (int j = 0; j < G4; ++j) {
    const float z = s.dz[j];
    acc0 = fmaf(z, w0[j], acc0);
    acc1 = fmaf(z, w1[j], acc1);
  }
  if (r0 < nr) s.din[r0] = acc0;
  if (r1 < nr) s.din[r1] = acc1;
  __syncwarp();
  return dct * gf;
}

// ------------------------------------------------------------------------------------------------
// forward of many sequences (predict / evaluate of the many-to-many network, and the one-to-one
// network when x_repeat != 0): warp per sample.  X [S][T][D] (or [S][D] repeated T times), out [S][T]
// logits (or [S] = the last step's logit when last_only).
template <bool EXT>
__global__ void __launch_bounds__(256)
lstm_forward_kernel(const LstmDesc d, const float *__restrict__ params, const float *__restrict__ X, int S,
                    int T, int x_repeat, float mask_value, int use_mask, int last_only, float *__restrict__ out) {
  extern __shared__ __align__(16) float sm[];
  float *ws = sm;
  stage_weights(d, params, ws);
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  const int sf = strip_floats(d, T, false);
  Strip s = carve_strip(d, sm + ((d.s_total + 3) & ~3) + warp * sf);
  const int U = d.U;
  for (int smp = blockIdx.x * nw + warp; smp < S; smp += gridDim.x * nw) {
    float c[LSTM_MAX_LAYERS];
#pragma unroll
    for (int l = 0; l < LSTM_MAX_LAYERS; ++l) c[l] = 0.f;
    for (int k = lane; k < d.L * U; k += 32) s.h[k] = 0.f;
    __syncwarp();
    for (int t = 0; t < T; ++t) {
      const float *xt = x_repeat ? X + (size_t)smp * d.D : X + ((size_t)smp * T + t) * d.D;
      int differs = 0;
      for (int k = lane; k < d.D; k += 32) { const float v = xt[k]; s.xin[k] = v; differs |= (v != mask_value); }
      const bool live = !use_mask || __any_sync(0xffffffffu, differs);
      __syncwarp();
      stack_forward<EXT>(d, ws, s, c, t, live, false, lane);
      if (!last_only || t == T - 1) {
        float u = lane < U ? s.h[(d.L - 1) * U + lane] * ws[d.s_wd + lane] : 0.f;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) u += __shfl_xor_sync(0xffffffffu, u, o);
        if (lane == 0) out[last_only ? smp : (size_t)smp * T + t] = u + ws[d.s_bd];
      }
      __syncwarp();
    }
  }
}

// value f = T(sign * u(x)) and df/dx of the one-to-one network with T steps (x repeated): warp per point
template <bool EXT>
__global__ void __launch_bounds__(128)
lstm_value_grad_kernel(const LstmDesc d, const float *__restrict__ params, const void *__restrict__ Xv, int x_is_f64,
                       int S, int T, int transform, float sign, const int *__restrict__ flags,
                       float *__restrict__ f_out, float *__restrict__ g_out) {
  extern __shared__ __align__(16) float sm[];
  float *ws = sm;
  stage_weights(d, params, ws);
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  const int sf = strip_floats(d, T, true);
  Strip s = carve_strip(d, sm + ((d.s_total + 3) & ~3) + warp * sf);
  const int U = d.U, L = d.L;
  for (int smp = blockIdx.x * nw + warp; smp < S; smp += gridDim.x * nw) {
    if (flags && !flags[smp]) continue;
    float c[LSTM_MAX_LAYERS];
#pragma unroll
    for (int l = 0; l < LSTM_MAX_LAYERS; ++l) c[l] = 0.f;
    for (int k = lane; k < L * U; k += 32) s.h[k] = 0.f;
    // fp64 trial points are rounded to fp32 here, as the Keras model casts its float64 input
    // (bore/decorators.py:73 hands TF the float64 array)
    if (x_is_f64) {
      const double *x = (const double *)Xv + (size_t)smp * d.D;
      for (int k = lane; k < d.D; k += 32) s.xin[k] = (float)x[k];
    } else {
      const float *x = (const float *)Xv + (size_t)smp * d.D;
      for (int k = lane; k < d.D; k += 32) s.xin[k] = x[k];
    }
    __syncwarp();
    for (int t = 0; t < T; ++t) stack_forward<EXT>(d, ws, s, c, t, true, true, lane);
    float u = lane < U ? s.h[(L - 1) * U + lane] * ws[d.s_wd + lane] : 0.f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) u += __shfl_xor_sync(0xffffffffu, u, o);
    u += ws[d.s_bd];
    const float v = sign * u;
    float fval, dT;
    if (transform == BORE_TRANSFORM_SIGMOID) { fval = 1.f / (1.f + expf(-v)); dT = fval * (1.f - fval); }
    else if (transform == BORE_TRANSFORM_EXP) { fval = expf(v); dT = fval; }
    else { fval = v; dT = 1.f; }
    const float du = dT * sign;
    float dh[LSTM_MAX_LAYERS], dc[LSTM_MAX_LAYERS];
#pragma unroll
    for (int l = 0; l < LSTM_MAX_LAYERS; ++l) { dh[l] = 0.f; dc[l] = 0.f; }
    float gx0 = 0.f;  // input gradient of coordinate `lane` (D <= 32), summed over the steps
    for (int t = T - 1; t >= 0; --t) {
      float dabove = (t == T - 1 && lane < U) ? du * ws[d.s_wd + lane] : 0.f;  // the Dense layer sees the last step
      for (int l = L - 1; l >= 0; --l) {
        const int in = in_dim(d, l);
        const float dcp = cell_backward<EXT>(d, ws, s, t, l, dh[l] + dabove, dc[l], lane);
        dh[l] = lane < U ? s.din[in + lane] : 0.f;
        dc[l] = dcp;
        dabove = (l > 0 && lane < U) ? s.din[lane] : 0.f;
        if (l == 0 && lane < d.D) gx0 += s.din[lane];
        __syncwarp();
      }
    }
    if (lane == 0) f_out[smp] = fval;
    if (lane < d.D) g_out[(size_t)smp * d.D + lane] = gx0;
    __syncwarp();
  }
}

// ------------------------------------------------------------------------------------------------
struct LstmFitArgs {
  LstmDesc d;
  float *params, *adam_m, *adam_v;
  long long t0;
  const float *X;       // [N][T][D]
  const float *Y;       // [N][T]
  int N, T, batch, epochs;
  int sample_warps;     // warps that carve a BPTT strip and run phase 1 (<= 8, as many as shared memory holds)
  const int *perm;      // [epochs][N]
  float mask_value;
  OptHyper opt;
  float l2[3 * LSTM_MAX_LAYERS + 2], l1[3 * LSTM_MAX_LAYERS + 2];
  float *loss_out;      // [epochs]
  float *scratch;       // A [L][T][B][AW] | Z [L][T][B][4U] | HT [T][B][U] | DU [T][B]
  float *opt_cache;     // Nadam's momentum cache (1 float)
  LrSchedule sched;
};

// OPT: the optimizers other than Adam (opt.cuh), the learning-rate schedules and the l1 regulariser terms; the Adam
// build keeps its own IEEE arithmetic
template <bool EXT, bool OPT>
__global__ void __launch_bounds__(256) lstm_fit_kernel(const LstmFitArgs a) {
  extern __shared__ __align__(16) float sm[];
  const LstmDesc &d = a.d;
  const int U = d.U, L = d.L, T = a.T, G4 = 4 * U, D = d.D;
  const int AW = (D > U ? D : U) + U;  // row width of A (cells with a narrower input leave a tail)
  const int B = a.batch;
  float *ws = sm;
  stage_weights(d, a.params, ws);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, nw = blockDim.x >> 5;
  const int sf = strip_floats(d, T, true);
  float *warp_area = sm + ((d.s_total + 3) & ~3);
  Strip s = carve_strip(d, warp_area + warp * sf);
  // staging tiles of the weight GEMMs alias the warps' strips (dead in that phase)
  float *tA = warp_area, *tZ = warp_area + LSTM_MAX_BATCH * AW;
  __shared__ float s_red[8];
  __shared__ float s_loss;
  float *gA = a.scratch;
  float *gZ = gA + (size_t)L * T * B * AW;
  float *gH = gZ + (size_t)L * T * B * G4;
  float *gU = gH + (size_t)T * B * U;
  const int spe = (a.N + B - 1) / B;
  OptRun<OPT> run(a.opt, a.t0, a.opt_cache);
  __syncthreads();

  for (int ep = 0; ep < a.epochs; ++ep) {
    float tot = 0.f;  // (thread 0) sum of batch loss * batch size, fp32 like the Keras metric
    for (int st = 0; st < spe; ++st) {
      const int s0 = st * B, nb = min(B, a.N - s0);
      const float inv_n = 1.f / (float)(nb * T);
      float lsum = 0.f;
      // ---- phase 1: forward + BPTT, warp per sample (the warps without a strip add 0 to the loss) ----
      for (int b = warp; warp < a.sample_warps && b < nb; b += a.sample_warps) {
        const int row = a.perm[(size_t)ep * a.N + s0 + b];
        const float *xs = a.X + (size_t)row * T * D;
        const float *ys = a.Y + (size_t)row * T;
        float c[LSTM_MAX_LAYERS];
#pragma unroll
        for (int l = 0; l < LSTM_MAX_LAYERS; ++l) c[l] = 0.f;
        for (int k = lane; k < L * U; k += 32) s.h[k] = 0.f;
        __syncwarp();
        unsigned live_mask = 0;
        float du_t[LSTM_MAX_STEPS];
        for (int t = 0; t < T; ++t) {
          int differs = 0;
          for (int k = lane; k < D; k += 32) { const float v = xs[t * D + k]; s.xin[k] = v; differs |= (v != a.mask_value); }
          const bool live = __any_sync(0xffffffffu, differs);
          if (live) live_mask |= 1u << t;
          __syncwarp();
          stack_forward<EXT>(d, ws, s, c, t, live, true, lane);
          float u = lane < U ? s.h[(L - 1) * U + lane] * ws[d.s_wd + lane] : 0.f;
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) u += __shfl_xor_sync(0xffffffffu, u, o);
          u += ws[d.s_bd];
          const float y = ys[t];
          // mean BCE on the logit, weight = mask, divided by batch x steps
          const float w = live ? 1.f : 0.f;
          lsum += w * (fmaxf(u, 0.f) - u * y + log1pf(expf(-fabsf(u))));
          du_t[t] = w * (l_sigmoid(u) - y) * inv_n;
          // top cell's output of this step and du for the Dense gradients
          if (lane < U) gH[((size_t)t * B + b) * U + lane] = s.h[(L - 1) * U + lane];
          if (lane == 0) gU[(size_t)t * B + b] = du_t[t];
          __syncwarp();
        }
        float dh[LSTM_MAX_LAYERS], dc[LSTM_MAX_LAYERS];
#pragma unroll
        for (int l = 0; l < LSTM_MAX_LAYERS; ++l) { dh[l] = 0.f; dc[l] = 0.f; }
        for (int t = T - 1; t >= 0; --t) {
          const bool live = (live_mask >> t) & 1u;
          if (!live) {  // h_t = h_{t-1}, c_t = c_{t-1}: the gradients pass through; nothing for the GEMMs
            for (int l = 0; l < L; ++l) {
              float *Zr = gZ + (((size_t)l * T + t) * B + b) * G4;
              float *Ar = gA + (((size_t)l * T + t) * B + b) * AW;
              for (int j = lane; j < G4; j += 32) Zr[j] = 0.f;
              for (int k = lane; k < AW; k += 32) Ar[k] = 0.f;
            }
            continue;
          }
          // h_{t-1} of every cell = its output at the last LIVE step before t (kept o * act(c)), else 0
          __syncwarp();
          for (int l = 0; l < L; ++l)
            if (lane < U) {
              float hv = 0.f;
              for (int tp = t - 1; tp >= 0; --tp)
                if ((live_mask >> tp) & 1u) {
                  const float *aa = s.acts + ((size_t)(tp * L + l) * 6) * U + lane;
                  hv = aa[3 * U] * aa[4 * U];
                  break;
                }
              s.h[l * U + lane] = hv;
            }
          for (int k = lane; k < D; k += 32) s.xin[k] = xs[t * D + k];
          __syncwarp();
          float dabove = lane < U ? du_t[t] * ws[d.s_wd + lane] : 0.f;  // TimeDistributed(Dense) at this step
          for (int l = L - 1; l >= 0; --l) {
            const int in = in_dim(d, l);
            const float dcp = cell_backward<EXT>(d, ws, s, t, l, dh[l] + dabove, dc[l], lane);
            // rows for the weight GEMMs: [input of the cell at step t ; h_{t-1}] and dz
            float *Zr = gZ + (((size_t)l * T + t) * B + b) * G4;
            float *Ar = gA + (((size_t)l * T + t) * B + b) * AW;
            for (int j = lane; j < G4; j += 32) Zr[j] = s.dz[j];
            if (l == 0) {
              for (int k = lane; k < in; k += 32) Ar[k] = s.xin[k];
            } else if (lane < U) {  // input = h_t of the cell below = o * act(c) kept at step t
              const float *ab = s.acts + ((size_t)(t * L + l - 1) * 6) * U + lane;
              Ar[lane] = ab[3 * U] * ab[4 * U];
            }
            for (int k = lane; k < U; k += 32) Ar[in + k] = s.h[l * U + k];
            for (int k = in + U + lane; k < AW; k += 32) Ar[k] = 0.f;
            dh[l] = lane < U ? s.din[in + lane] : 0.f;
            dc[l] = dcp;
            dabove = (l > 0 && lane < U) ? s.din[lane] : 0.f;
            __syncwarp();
          }
        }
      }
      // ---- loss of the batch ----
      // (every lane of a warp accumulated the same per-sample terms: take lane 0's)
      if (lane == 0) s_red[warp] = lsum;
      __syncthreads();
      if (tid == 0) {
        float ls = 0.f;
        for (int w2 = 0; w2 < nw; ++w2) ls += s_red[w2];
        s_loss = ls * inv_n;
      }
      // ---- phase 2: weight gradients as small GEMMs + Adam ----
      OptStep os;
      float alpha = 0.f;
      if (OPT) {
        os = run.step(a.opt, a.sched);
      } else {
        run.t += 1;
        run.p1 *= (double)a.opt.b1; run.p2 *= (double)a.opt.b2;
        alpha = (float)((double)a.opt.lr * sqrt(1.0 - run.p2) / (1.0 - run.p1));
      }
      const float omb1 = 1.f - a.opt.b1, omb2 = 1.f - a.opt.b2;
      float reg = 0.f;  // this thread's share of the l1 / l2 penalty (value, for the reported loss)
      auto adam = [&](int pi, float g, int ra) {  // ra: the parameter's array, Keras order
        const float wv = a.params[pi];
        regularize(OPT ? a.l1[ra] : 0.f, a.l2[ra], wv, reg, g);
        float mm = a.adam_m[pi], vv = a.adam_v[pi];
        if (OPT) {
          const float wn = opt_update<true>(a.opt, os, wv, g, mm, vv);
          a.adam_m[pi] = mm; a.adam_v[pi] = vv;
          a.params[pi] = wn;
          return wn;
        }
        mm += (g - mm) * omb1;
        vv += (g * g - vv) * omb2;
        a.adam_m[pi] = mm; a.adam_v[pi] = vv;
        const float wn = wv - (mm * alpha) / (sqrtf(vv) + a.opt.eps);
        a.params[pi] = wn;
        return wn;
      };
      const int j = tid & 127, half = tid >> 7;     // column of the gate matrix, half of the rows
      for (int l = 0; l < L; ++l) {
        const int in = in_dim(d, l), nr = in + U;
        const int KH = (nr + 1) / 2;                // rows per half (<= 32)
        float acc[32];
#pragma unroll
        for (int q = 0; q < 32; ++q) acc[q] = 0.f;
        float accb = 0.f;
        for (int t = 0; t < T; ++t) {
          __syncthreads();  // the tiles (and, first time, the strips they alias) are free
          const float *srcA = gA + ((size_t)l * T + t) * B * AW;
          const float *srcZ = gZ + ((size_t)l * T + t) * B * G4;
          for (int e = tid; e < nb * AW; e += blockDim.x) tA[e] = srcA[e];
          for (int e = tid; e < nb * G4; e += blockDim.x) tZ[e] = srcZ[e];
          __syncthreads();
          if (j < G4) {
            for (int b = 0; b < nb; ++b) {
              const float z = tZ[b * G4 + j];
              const float *ar = tA + b * AW + half * KH;
              accb += z;
#pragma unroll
              for (int q = 0; q < 32; ++q)
                if (q < KH) acc[q] = fmaf(ar[q], z, acc[q]);
            }
          }
        }
        if (j < G4) {
          float *Wimg = ws + d.s_w[l];
          const int LD = ldw(d);
#pragma unroll
          for (int q = 0; q < 32; ++q) {
            const int k = half * KH + q;
            if (q < KH && k < nr) {
              const bool isK = k < in;
              const int pi = isK ? d.k_off[l] + k * G4 + j : d.r_off[l] + (k - in) * G4 + j;
              const float wn = adam(pi, acc[q], 3 * l + (isK ? 0 : 1));
              Wimg[k * LD + j] = wn;
            }
          }
          if (half == 0) ws[d.s_b[l] + j] = adam(d.b_off[l] + j, accb, 3 * l + 2);
        }
      }
      // Dense layer: dWd[k] = sum_{t,b} h_top[t][b][k] du[t][b]; dbd = sum du  (warp 0, lane = k)
      if (warp == 0) {
        float gk = 0.f, gb = 0.f;
        for (int t = 0; t < T; ++t)
          for (int b = 0; b < nb; ++b) {
            const float du = gU[(size_t)t * B + b];
            gb += du;
            if (lane < U) gk = fmaf(gH[((size_t)t * B + b) * U + lane], du, gk);
          }
        if (lane < U) ws[d.s_wd + lane] = adam(d.wd_off + lane, gk, 3 * L);
        if (lane == 0) ws[d.s_bd] = adam(d.bd_off, gb, 3 * L + 1);
      }
      // regulariser penalty into the reported loss (values BEFORE this step's update)
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) reg += __shfl_xor_sync(0xffffffffu, reg, o);
      __syncthreads();
      if (lane == 0) s_red[warp] = reg;
      __syncthreads();
      if (tid == 0) {
        float r = 0.f;
        for (int w2 = 0; w2 < nw; ++w2) r += s_red[w2];
        tot += (s_loss + r) * (float)nb;
      }
      __syncthreads();
    }
    if (tid == 0) a.loss_out[ep] = tot / (float)a.N;
  }
  if (OPT && tid == 0) *a.opt_cache = run.cache;
}

// evaluate(): masked BCE-with-logits of precomputed logits [N][T] divided by N x T (+ the l1 / l2 penalty),
// and Keras' binary_accuracy on the LOGIT (threshold 0.5, the from_logits quirk -- logging only)
// averaged over the unmasked steps.  One CTA, fixed summation order.  out[0] = loss, out[1] = accuracy.
__global__ void __launch_bounds__(256)
lstm_evaluate_kernel(const LstmDesc d, const float *__restrict__ params, const float *__restrict__ l2,
                     const float *__restrict__ l1,
                     const float *__restrict__ X, const float *__restrict__ Y, const float *__restrict__ logits,
                     int N, int T, float mask_value, float *__restrict__ out) {
  __shared__ float red[3][8];
  float ls = 0.f, hit = 0.f, cnt = 0.f;
  for (int e = threadIdx.x; e < N * T; e += blockDim.x) {
    const float *x = X + (size_t)e * d.D;
    bool live = false;
    for (int k = 0; k < d.D; ++k) live |= (x[k] != mask_value);
    if (!live) continue;
    const float u = logits[e], y = Y[e];
    ls += fmaxf(u, 0.f) - u * y + log1pf(expf(-fabsf(u)));
    hit += ((u > 0.5f ? 1.f : 0.f) == y) ? 1.f : 0.f;
    cnt += 1.f;
  }
  float reg = 0.f;
  for (int a = 0; a < 3 * d.L + 2; ++a) {
    const float f = l2[a], f1 = l1[a];
    if (f == 0.f && f1 == 0.f) continue;
    const int l = a / 3, r = a - 3 * l;
    int off, n;
    if (a == 3 * d.L) { off = d.wd_off; n = d.U; }
    else if (a == 3 * d.L + 1) { off = d.bd_off; n = 1; }
    else if (r == 0) { off = d.k_off[l]; n = in_dim(d, l) * 4 * d.U; }
    else if (r == 1) { off = d.r_off[l]; n = d.U * 4 * d.U; }
    else { off = d.b_off[l]; n = 4 * d.U; }
    for (int e = threadIdx.x; e < n; e += blockDim.x) {
      const float w = params[off + e];
      if (f != 0.f) reg += f * w * w;
      if (f1 != 0.f) reg += f1 * fabsf(w);
    }
  }
  ls = ls / (float)(N * T) + reg;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ls += __shfl_xor_sync(0xffffffffu, ls, o);
    hit += __shfl_xor_sync(0xffffffffu, hit, o);
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { red[0][warp] = ls; red[1][warp] = hit; red[2][warp] = cnt; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f, b = 0.f, c = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { a += red[0][w]; b += red[1][w]; c += red[2][w]; }
    out[0] = a;
    out[1] = c > 0.f ? b / c : 0.f;
  }
}

int make_desc(int D, int U, int L, int act, LstmDesc &d) {
  d.D = D; d.U = U; d.L = L; d.act = act;
  int off = 0, so = 0;
  for (int l = 0; l < L; ++l) {
    const int in = l == 0 ? D : U;
    d.k_off[l] = off; off += in * 4 * U;
    d.r_off[l] = off; off += U * 4 * U;
    d.b_off[l] = off; off += 4 * U;
    d.s_w[l] = so; so += (in + U) * (4 * U + 1);
    so = (so + 3) & ~3;
    d.s_b[l] = so; so += 4 * U;
  }
  d.wd_off = off; off += U;
  d.bd_off = off; off += 1;
  d.n_params = off;
  d.s_wd = so; so += U;
  d.s_bd = so; so += 1;
  d.s_total = so;
  return 0;
}

size_t fit_scratch_floats(const LstmDesc &d, int T, int B) {
  const int AW = (d.D > d.U ? d.D : d.U) + d.U;
  return (size_t)d.L * T * B * AW + (size_t)d.L * T * B * 4 * d.U + (size_t)T * B * d.U + (size_t)T * B;
}

// Warps of a launch in which every warp keeps a strip of `strip` floats beside the weight image: as many
// as 227 KB of shared memory holds, at most `max_warps`.  A net whose strips grow with steps and cells
// (four cells of 32 units at 8 steps) runs on fewer warps instead of being refused; at least one, so
// that a net not even one strip fits is refused by the launch's shared-memory check.
int warps_that_fit(const LstmDesc &d, int strip, int max_warps) {
  const int room = 227 * 1024 / (int)sizeof(float) - ((d.s_total + 3) & ~3);
  return std::max(1, std::min(max_warps, room / strip));
}

}  // namespace

extern "C" {

int bore_lstm_create(int input_dim, int units, int num_layers, int activation, int device, bore_lstm **out) {
  BORE_CHECK(out != nullptr, "bore_lstm_create: out is NULL");
  BORE_CHECK(input_dim >= 1 && input_dim <= LSTM_MAX_DIM, "bore_lstm_create: input_dim=%d outside [1,%d]",
             input_dim, LSTM_MAX_DIM);
  BORE_CHECK(units >= 1 && units <= LSTM_MAX_UNITS, "bore_lstm_create: units=%d outside [1,%d]", units,
             LSTM_MAX_UNITS);
  BORE_CHECK(num_layers >= 1 && num_layers <= LSTM_MAX_LAYERS, "bore_lstm_create: num_layers=%d outside [1,%d]",
             num_layers, LSTM_MAX_LAYERS);
  BORE_CHECK(activation >= BORE_ACT_LINEAR && activation <= BORE_ACT_EXPONENTIAL, "bore_lstm_create: unknown activation %d",
             activation);
  BORE_CHECK(bore_device_count() > 0, "bore_lstm_create: no CUDA device visible -- bore_b200 has no CPU fallback");
  BORE_CUDA(cudaSetDevice(device));
  bore_lstm *h = new bore_lstm();
  memset(h, 0, sizeof(*h));
  make_desc(input_dim, units, num_layers, activation, h->desc);
  h->device = device;
  cudaDeviceProp prop;
  BORE_CUDA(cudaGetDeviceProperties(&prop, device));
  h->sm_count = prop.multiProcessorCount;
  h->opt = OptHyper{1e-3f, 0.9f, 0.999f, 1e-7f, 0.f, 0.f, BORE_OPT_ADAM, 0};  // Keras "adam"
  const size_t nb = (size_t)h->desc.n_params * sizeof(float);
  BORE_CUDA(cudaMalloc(&h->params, nb));
  BORE_CUDA(cudaMalloc(&h->adam_m, nb));
  BORE_CUDA(cudaMalloc(&h->adam_v, nb));
  BORE_CUDA(cudaMalloc(&h->opt_cache, sizeof(float)));
  BORE_CUDA(cudaMemset(h->params, 0, nb));
  BORE_CHECK_RC(opt_reset_state(h->opt, h->adam_m, h->adam_v, h->desc.n_params, nullptr, h->opt_cache, 1, 0));
  BORE_CUDA(cudaDeviceSynchronize());
  *out = h;
  return 0;
}

int bore_lstm_destroy(bore_lstm *h) {
  if (!h) return 0;
  cudaSetDevice(h->device);
  cudaFree(h->params); cudaFree(h->adam_m); cudaFree(h->adam_v); cudaFree(h->opt_cache);
  if (h->scratch) cudaFree(h->scratch);
  delete h;
  return 0;
}

int bore_lstm_num_params(const bore_lstm *h) { return h ? h->desc.n_params : -1; }

int bore_lstm_set_weights(bore_lstm *h, const float *params_host) {
  BORE_CHECK(h && params_host, "NULL argument");
  BORE_CUDA(cudaSetDevice(h->device));
  BORE_CUDA(cudaDeviceSynchronize());
  BORE_CUDA(cudaMemcpy(h->params, params_host, (size_t)h->desc.n_params * sizeof(float), cudaMemcpyHostToDevice));
  return 0;
}

int bore_lstm_get_weights(bore_lstm *h, float *params_host) {
  BORE_CHECK(h && params_host, "NULL argument");
  BORE_CUDA(cudaSetDevice(h->device));
  BORE_CUDA(cudaDeviceSynchronize());
  BORE_CUDA(cudaMemcpy(params_host, h->params, (size_t)h->desc.n_params * sizeof(float), cudaMemcpyDeviceToHost));
  return 0;
}

int bore_lstm_set_adam_state(bore_lstm *h, const float *m_host, const float *v_host, int64_t iterations) {
  BORE_CHECK(h && m_host && v_host, "NULL argument");
  BORE_CUDA(cudaSetDevice(h->device));
  BORE_CUDA(cudaDeviceSynchronize());
  const size_t nb = (size_t)h->desc.n_params * sizeof(float);
  BORE_CUDA(cudaMemcpy(h->adam_m, m_host, nb, cudaMemcpyHostToDevice));
  BORE_CUDA(cudaMemcpy(h->adam_v, v_host, nb, cudaMemcpyHostToDevice));
  h->adam_t = iterations;
  return 0;
}

int bore_lstm_get_adam_state(bore_lstm *h, float *m_host, float *v_host, int64_t *iterations) {
  BORE_CHECK(h && m_host && v_host && iterations, "NULL argument");
  BORE_CUDA(cudaSetDevice(h->device));
  BORE_CUDA(cudaDeviceSynchronize());
  const size_t nb = (size_t)h->desc.n_params * sizeof(float);
  BORE_CUDA(cudaMemcpy(m_host, h->adam_m, nb, cudaMemcpyDeviceToHost));
  BORE_CUDA(cudaMemcpy(v_host, h->adam_v, nb, cudaMemcpyDeviceToHost));
  *iterations = h->adam_t;
  return 0;
}

int bore_lstm_set_optimizer_kind(bore_lstm *h, int kind, const float *hp) {
  OptHyper o;
  BORE_CHECK_RC(opt_from_array(kind, hp, o, "bore_lstm_set_optimizer_kind"));
  BORE_CHECK(h != nullptr, "NULL handle");
  BORE_CUDA(cudaSetDevice(h->device));
  if (o.kind != h->opt.kind) {  // a new optimizer starts from fresh slots, as Keras builds them
    BORE_CUDA(cudaDeviceSynchronize());
    BORE_CHECK_RC(opt_reset_state(o, h->adam_m, h->adam_v, h->desc.n_params, nullptr, h->opt_cache, 1, 0));
    BORE_CUDA(cudaDeviceSynchronize());
    h->adam_t = 0;
  }
  h->opt = o;
  return 0;
}

int bore_lstm_set_lr_schedule(bore_lstm *h, int kind, const float *sp, int n_sp) {
  LrSchedule s;
  BORE_CHECK_RC(lr_schedule_from_array(kind, sp, n_sp, s, "bore_lstm_set_lr_schedule"));
  BORE_CHECK(h != nullptr, "NULL handle");
  h->sched = s;  // the state is kept, as Keras keeps its slots under a new rate
  return 0;
}

int bore_lstm_get_nadam_cache(bore_lstm *h, float *cache_host) {
  BORE_CHECK(h && cache_host, "NULL argument");
  BORE_CUDA(cudaSetDevice(h->device));
  BORE_CUDA(cudaDeviceSynchronize());
  BORE_CUDA(cudaMemcpy(cache_host, h->opt_cache, sizeof(float), cudaMemcpyDeviceToHost));
  return 0;
}

int bore_lstm_set_nadam_cache(bore_lstm *h, float cache) {
  BORE_CHECK(h != nullptr, "NULL handle");
  BORE_CUDA(cudaSetDevice(h->device));
  BORE_CUDA(cudaDeviceSynchronize());
  BORE_CUDA(cudaMemcpy(h->opt_cache, &cache, sizeof(float), cudaMemcpyHostToDevice));
  return 0;
}

int bore_lstm_set_regularizers(bore_lstm *h, const float *l2_host) {
  BORE_CHECK(h && l2_host, "NULL argument");
  for (int i = 0; i < 3 * h->desc.L + 2; ++i) {
    BORE_CHECK(l2_host[i] >= 0.f, "negative l2 factor");
    h->l2[i] = l2_host[i];
  }
  return 0;
}

int bore_lstm_set_l1_regularizers(bore_lstm *h, const float *l1_host) {
  BORE_CHECK(h && l1_host, "NULL argument");
  const int n = 3 * h->desc.L + 2;
  for (int i = 0; i < n; ++i)
    BORE_CHECK(isfinite(l1_host[i]) && l1_host[i] >= 0.f, "l1 factor %d is %g: it must be finite and >= 0", i,
               (double)l1_host[i]);
  for (int i = 0; i < n; ++i) h->l1[i] = l1_host[i];
  return 0;
}

// logits of the many-to-many network: X_dev [S][T][D] -> out_dev [S][T]; with use_mask the steps
// whose features all equal mask_value are masked (Masking layer).
int bore_lstm_predict_sequences(bore_lstm *h, const float *X_dev, int S, int T, float mask_value, int use_mask,
                                float *out_dev, void *stream) {
  BORE_NVTX("bore:lstm predict (K7)");
  BORE_CHECK(h && X_dev && out_dev, "NULL argument");
  BORE_CHECK(S >= 0 && T >= 1 && T <= LSTM_MAX_STEPS, "bore_lstm_predict_sequences: S=%d, T=%d (max %d steps)", S, T,
             LSTM_MAX_STEPS);
  if (S == 0) return 0;
  BORE_CUDA(cudaSetDevice(h->device));
  const int warps = 8;
  const size_t smem = ((size_t)((h->desc.s_total + 3) & ~3) + (size_t)warps * strip_floats(h->desc, T, false)) * sizeof(float);
  const auto kernel = acts_ext(&h->desc.act, 1) ? lstm_forward_kernel<true> : lstm_forward_kernel<false>;
  BORE_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int grid = std::min((S + warps - 1) / warps, h->sm_count * 2);
  kernel<<<grid, warps * 32, smem, (cudaStream_t)stream>>>(h->desc, h->params, X_dev, S, T, 0, mask_value, use_mask, 0,
                                                          out_dev);
  BORE_CUDA(cudaGetLastError());
  return 0;
}

// the one-to-one network with num_steps steps (RepeatVector): X_dev [S][D] -> out_dev [S]
int bore_lstm_predict(bore_lstm *h, const float *X_dev, int S, int num_steps, float *out_dev, void *stream) {
  BORE_NVTX("bore:lstm predict one-to-one (K7)");
  BORE_CHECK(h && X_dev && out_dev, "NULL argument");
  BORE_CHECK(S >= 0 && num_steps >= 1 && num_steps <= LSTM_MAX_STEPS, "bore_lstm_predict: S=%d, num_steps=%d", S,
             num_steps);
  if (S == 0) return 0;
  BORE_CUDA(cudaSetDevice(h->device));
  const int warps = 8;
  const size_t smem = ((size_t)((h->desc.s_total + 3) & ~3) + (size_t)warps * strip_floats(h->desc, num_steps, false)) * sizeof(float);
  const auto kernel = acts_ext(&h->desc.act, 1) ? lstm_forward_kernel<true> : lstm_forward_kernel<false>;
  BORE_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int grid = std::min((S + warps - 1) / warps, h->sm_count * 2);
  kernel<<<grid, warps * 32, smem, (cudaStream_t)stream>>>(h->desc, h->params, X_dev, S, num_steps, 1, 0.f, 0, 1,
                                                          out_dev);
  BORE_CUDA(cudaGetLastError());
  return 0;
}

// f = T(+-u(x)), g = df/dx of the one-to-one network for every row of X_dev [S][D] (those with
// flags_dev[i] != 0 when flags_dev is given): the convert() closure of bore/base.py:35-42.
int bore_lstm_value_and_grad(bore_lstm *h, int num_steps, int transform, int negate, const void *X_dev,
                             int x_is_f64, int S, const int32_t *flags_dev, float *f_dev, float *g_dev,
                             void *stream) {
  BORE_NVTX("bore:lstm value_and_grad (K7)");
  BORE_CHECK(h && X_dev && f_dev && g_dev, "NULL argument");
  BORE_CHECK(S >= 0 && num_steps >= 1 && num_steps <= LSTM_MAX_STEPS, "bore_lstm_value_and_grad: S=%d, num_steps=%d",
             S, num_steps);
  BORE_CHECK(transform >= 0 && transform <= BORE_TRANSFORM_EXP, "unknown transform code %d", transform);
  if (S == 0) return 0;
  BORE_CUDA(cudaSetDevice(h->device));
  const int sf = strip_floats(h->desc, num_steps, true);
  const int warps = warps_that_fit(h->desc, sf, 4);
  const size_t smem = ((size_t)((h->desc.s_total + 3) & ~3) + (size_t)warps * sf) * sizeof(float);
  BORE_CHECK(smem <= 227 * 1024, "bore_lstm_value_and_grad: needs %zu B of shared memory", smem);
  const auto kernel = acts_ext(&h->desc.act, 1) ? lstm_value_grad_kernel<true> : lstm_value_grad_kernel<false>;
  BORE_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int grid = std::min((S + warps - 1) / warps, h->sm_count * 2);
  kernel<<<grid, warps * 32, smem, (cudaStream_t)stream>>>(
      h->desc, h->params, X_dev, x_is_f64, S, num_steps, transform, negate ? -1.f : 1.f, flags_dev, f_dev, g_dev);
  BORE_CUDA(cudaGetLastError());
  return 0;
}

// Keras fit on padded sequences: X_dev [N][T][D], Y_dev [N][T] (fp32), perm_dev [epochs][N] int32,
// loss_dev [epochs].  Asynchronous on `stream`; weights and Adam state updated in place.
int bore_lstm_fit(bore_lstm *h, const float *X_dev, const float *Y_dev, int N, int T, float mask_value,
                  int batch_size, int epochs, const int32_t *perm_dev, float *loss_dev, void *stream) {
  BORE_NVTX("bore:lstm fit (K7)");
  BORE_CHECK(h && X_dev && Y_dev && perm_dev && loss_dev, "NULL argument");
  BORE_CHECK(N >= 1 && T >= 1 && T <= LSTM_MAX_STEPS, "bore_lstm_fit: N=%d, T=%d (max %d steps)", N, T, LSTM_MAX_STEPS);
  BORE_CHECK(batch_size >= 1 && batch_size <= LSTM_MAX_BATCH, "bore_lstm_fit: batch_size=%d outside [1,%d]", batch_size,
             LSTM_MAX_BATCH);
  BORE_CHECK(epochs >= 0, "bore_lstm_fit: epochs=%d", epochs);
  if (epochs == 0) return 0;
  BORE_CUDA(cudaSetDevice(h->device));
  const size_t need = fit_scratch_floats(h->desc, T, batch_size) * sizeof(float);
  if (h->scratch_bytes < need) {
    if (h->scratch) BORE_CUDA(cudaFree(h->scratch));
    h->scratch = nullptr; h->scratch_bytes = 0;
    BORE_CUDA(cudaMalloc(&h->scratch, need));
    h->scratch_bytes = need;
  }
  LstmFitArgs a;
  a.d = h->desc;
  a.params = h->params; a.adam_m = h->adam_m; a.adam_v = h->adam_v;
  a.t0 = h->adam_t;
  a.X = X_dev; a.Y = Y_dev; a.N = N; a.T = T; a.batch = batch_size; a.epochs = epochs;
  a.perm = perm_dev; a.mask_value = mask_value;
  a.opt = h->opt; a.opt_cache = h->opt_cache; a.sched = h->sched;
  for (int i = 0; i < 3 * LSTM_MAX_LAYERS + 2; ++i) { a.l2[i] = h->l2[i]; a.l1[i] = h->l1[i]; }
  a.loss_out = loss_dev;
  a.scratch = h->scratch;
  // 256 threads whatever the number of sample warps: phase 2's GEMM mapping takes all of them
  const int warps = 8;
  const int sf = strip_floats(h->desc, T, true);
  a.sample_warps = warps_that_fit(h->desc, sf, warps);
  const int AW = (h->desc.D > h->desc.U ? h->desc.D : h->desc.U) + h->desc.U;
  const size_t strips = (size_t)a.sample_warps * sf;
  const size_t tiles = (size_t)LSTM_MAX_BATCH * (AW + 4 * h->desc.U);
  const size_t smem = ((size_t)((h->desc.s_total + 3) & ~3) + std::max(strips, tiles)) * sizeof(float);
  BORE_CHECK(smem <= 227 * 1024, "bore_lstm_fit: needs %zu B of shared memory", smem);
  bool any_l1 = false;
  for (int i = 0; i < 3 * LSTM_MAX_LAYERS + 2; ++i) any_l1 = any_l1 || h->l1[i] != 0.f;
  const auto kernel = with_flags([](auto e, auto o) { return lstm_fit_kernel<e, o>; }, acts_ext(&h->desc.act, 1),
                                 opt_build(h->opt, h->sched) || any_l1);
  BORE_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kernel<<<1, warps * 32, smem, (cudaStream_t)stream>>>(a);
  BORE_CUDA(cudaGetLastError());
  h->adam_t += (long long)epochs * ((N + batch_size - 1) / batch_size);
  return 0;
}

// Model.evaluate on padded sequences -> out_host[0] = loss (masked BCE / (N x T) + l1 / l2 terms),
// out_host[1] = accuracy over the unmasked steps (multi_fidelity.py:226).  Synchronises `stream`.
int bore_lstm_evaluate(bore_lstm *h, const float *X_dev, const float *Y_dev, int N, int T, float mask_value,
                       float *out_host, void *stream) {
  BORE_NVTX("bore:lstm evaluate (K7)");
  BORE_CHECK(h && X_dev && Y_dev && out_host, "NULL argument");
  BORE_CHECK(N >= 1 && T >= 1 && T <= LSTM_MAX_STEPS, "bore_lstm_evaluate: N=%d, T=%d (max %d steps)", N, T,
             LSTM_MAX_STEPS);
  BORE_CUDA(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  const int nl2 = 3 * LSTM_MAX_LAYERS + 2;
  float *buf = nullptr;  // logits [N][T] | l2 [nl2] | l1 [nl2] | out [2]
  BORE_CUDA(cudaMallocAsync(&buf, ((size_t)N * T + 2 * nl2 + 2) * sizeof(float), st));
  float *l2d = buf + (size_t)N * T, *l1d = l2d + nl2, *outd = l1d + nl2;
  BORE_CUDA(cudaMemcpyAsync(l2d, h->l2, nl2 * sizeof(float), cudaMemcpyHostToDevice, st));
  BORE_CUDA(cudaMemcpyAsync(l1d, h->l1, nl2 * sizeof(float), cudaMemcpyHostToDevice, st));
  int rc = bore_lstm_predict_sequences(h, X_dev, N, T, mask_value, 1, buf, stream);
  if (rc == 0) {
    lstm_evaluate_kernel<<<1, 256, 0, st>>>(h->desc, h->params, l2d, l1d, X_dev, Y_dev, buf, N, T, mask_value, outd);
    BORE_CUDA(cudaGetLastError());
    BORE_CUDA(cudaMemcpyAsync(out_host, outd, 2 * sizeof(float), cudaMemcpyDeviceToHost, st));
    BORE_CUDA(cudaStreamSynchronize(st));
  }
  BORE_CUDA(cudaFreeAsync(buf, st));
  return rc;
}

}  // extern "C"
